// Sampling, per-entity 4x4 composition and batched vertex transforms for sm_100a.
//
// Replaces (reference paths relative to the Fireflies tree):
//   fireflies/sampling/base.py:54-74, uniform.py:16-19, uniform_scalar_to_vec3.py:18-38,
//   gaussian_distribution.py:19-20, animation.py:27-45          -> ffb_sample, ffb_sample_anim_index
//   fireflies/utils/math.py:24-60,203-209; entity/base.py:194-244; entity/mesh.py:131-150
//                                                                -> ffb_compose_world
//   fireflies/utils/math.py:220-235; entity/mesh.py:158-165,183-198 -> ffb_transform_vertices/points(_bwd, _bwd_full)
//   fireflies/projection/laser.py:199-206,262-290                -> ffb_rays_to_ndc, ffb_clamp_to_fov
//
// The reference spends ~190 tiny aten ops and 12 host syncs per entity per sample (SURVEY.md 0-7); here a
// whole batch of B samples x E entities is two launches with no host round trip, and the vertex pass
// moves exactly 12 B in + 12 B out per vertex with 128-bit accesses.
#include "ffb_common.cuh"

namespace ffb {
namespace scene {

// ---- sampling ---------------------------------------------------------------------------------------
__device__ __forceinline__ float lerp_ref(float u, float a, float b) {
    // utils/math.py:174-175: rands * (b - a) + a  -- three separately rounded fp32 ops
    return __fadd_rn(__fmul_rn(u, __fsub_rn(b, a)), a);
}

__global__ void __launch_bounds__(256) sample_kernel(const ffb_sampler* __restrict__ samplers, int S, int B, int mode,
                                                     uint64_t seed, uint64_t sample0, const float* __restrict__ variates,
                                                     float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * S) return;
    const int b = i / S, s = i - b * S;
    const ffb_sampler sp = samplers[s];
    float v[3] = {0.f, 0.f, 0.f};
    float z[4];
    if (mode == FFB_MODE_INJECTED) {
        z[0] = variates[(size_t)i * 3]; z[1] = variates[(size_t)i * 3 + 1]; z[2] = variates[(size_t)i * 3 + 2]; z[3] = 0.f;
    } else {
        const uint64_t g = sample0 + (uint64_t)b;
        uint32_t r[4];
        Philox::gen(seed, (uint32_t)g, (uint32_t)(g >> 32), (uint32_t)s, 0x5A3D1E00u, r);
        if (sp.kind == FFB_SAMPLER_GAUSSIAN) {     // Box-Muller on two pairs
            const float u0 = ((float)(r[0] >> 8) + 1.0f) * (1.0f / 16777216.0f), u1 = Philox::u01(r[1]);
            const float u2 = ((float)(r[2] >> 8) + 1.0f) * (1.0f / 16777216.0f), u3 = Philox::u01(r[3]);
            const float ra = sqrtf(-2.0f * logf(u0)), rb = sqrtf(-2.0f * logf(u2));
            float sa, ca, sb, cb;
            sincospif(2.0f * u1, &sa, &ca);
            sincospif(2.0f * u3, &sb, &cb);
            z[0] = ra * ca; z[1] = ra * sa; z[2] = rb * cb; z[3] = rb * sb;
        } else {
            z[0] = Philox::u01(r[0]); z[1] = Philox::u01(r[1]); z[2] = Philox::u01(r[2]); z[3] = 0.f;
        }
    }
    const int dim = sp.dim < 1 ? 1 : (sp.dim > 3 ? 3 : sp.dim);
    if (sp.kind == FFB_SAMPLER_GAUSSIAN) {
        for (int k = 0; k < dim; ++k) v[k] = __fadd_rn(sp.mean[k], __fmul_rn(sp.std[k], z[k]));
    } else if (sp.kind == FFB_SAMPLER_SCALAR_TO_VEC3) {
        const float x = lerp_ref(z[0], sp.vmin[0], sp.vmax[0]);
        v[0] = v[1] = v[2] = x;
    } else {
        for (int k = 0; k < dim; ++k) v[k] = lerp_ref(z[k], sp.vmin[k], sp.vmax[k]);
    }
    out[(size_t)i * 3] = v[0]; out[(size_t)i * 3 + 1] = v[1]; out[(size_t)i * 3 + 2] = v[2];
}

// utils/math.py:170-175 for arbitrary shapes: out = u * (b - a) + a
__global__ void __launch_bounds__(256) uniform_between_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                              const float* __restrict__ u, long long n, float* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = lerp_ref(u[i], a[i], b[i]);
}

// Sampler.sample_eval (sampling/base.py:64-74) as a state machine, one thread per sampler walking the B
// successive calls.  Reproduces the reference's aliasing: the value returned is the post-increment
// _current_step; after the first wrap _current_step *is* _min_range, so stepping drifts vmin.
__global__ void __launch_bounds__(128) sample_eval_kernel(ffb_sampler* samplers, int S, int B, float* __restrict__ out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    ffb_sampler sp = samplers[s];
    const int dim = sp.dim < 1 ? 1 : (sp.dim > 3 ? 3 : sp.dim);
    for (int b = 0; b < B; ++b) {
        bool all_eq = true;
        for (int k = 0; k < dim; ++k) all_eq = all_eq && (sp.vmin[k] == sp.vmax[k]);
        float v[3] = {0.f, 0.f, 0.f};
        if (all_eq) {
            for (int k = 0; k < dim; ++k) v[k] = sp.vmin[k];
        } else {
            bool over = false;
            for (int k = 0; k < dim; ++k) {
                sp.cur[k] = __fadd_rn(sp.cur[k], sp.step);
                if (sp.aliased) sp.vmin[k] = sp.cur[k];
                v[k] = sp.cur[k];
                over = over || (sp.cur[k] > sp.vmax[k]);
            }
            if (over) {
                for (int k = 0; k < dim; ++k) sp.cur[k] = sp.vmin[k];
                sp.aliased = 1;
            }
        }
        if (sp.kind == FFB_SAMPLER_SCALAR_TO_VEC3) v[1] = v[2] = v[0];
        float* o = out + ((size_t)b * S + s) * 3;
        o[0] = v[0]; o[1] = v[1]; o[2] = v[2];
    }
    samplers[s] = sp;
}

__global__ void __launch_bounds__(128) anim_index_kernel(const int32_t* __restrict__ amin, const int32_t* __restrict__ amax,
                                                         int32_t* cur, int M, int B, int mode, uint64_t seed, uint64_t sample0,
                                                         int32_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (mode == FFB_MODE_EVAL) {       // sampling/animation.py:27-34 : sequential walk, max inclusive
        if (i >= M) return;
        int c = cur[i];
        for (int b = 0; b < B; ++b) {
            out[(size_t)b * M + i] = c;
            c += 1;
            if (c > amax[i]) c = amin[i];
        }
        cur[i] = c;
    } else {                           // sampling/animation.py:36-37 : randint(min, max-1)
        if (i >= B * M) return;
        const int b = i / M, m = i - b * M;
        const uint64_t g = sample0 + (uint64_t)b;
        uint32_t r[4];
        Philox::gen(seed, (uint32_t)g, (uint32_t)(g >> 32), (uint32_t)m, 0xA11A0001u, r);
        const int span = amax[m] - amin[m];
        out[i] = span > 0 ? amin[m] + (int)(((uint64_t)r[0] * (uint64_t)span) >> 32) : amin[m];
    }
}

// ---- compose ----------------------------------------------------------------------------------------
struct M4 { float m[16]; };

__device__ __forceinline__ M4 mul4(const M4& a, const M4& b) {
    M4 r;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float s = a.m[i * 4] * b.m[j];
            s = fmaf(a.m[i * 4 + 1], b.m[4 + j], s);
            s = fmaf(a.m[i * 4 + 2], b.m[8 + j], s);
            s = fmaf(a.m[i * 4 + 3], b.m[12 + j], s);
            r.m[i * 4 + j] = s;
        }
    return r;
}
__device__ __forceinline__ void mul3(const float* a, const float* b, float* r) {
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            float s = a[i * 3] * b[j];
            s = fmaf(a[i * 3 + 1], b[3 + j], s);
            s = fmaf(a[i * 3 + 2], b[6 + j], s);
            r[i * 3 + j] = s;
        }
}
// python math.cos/sin on the fp32 angle: fp64 trig, rounded to fp32 when the matrix tensor is built
__device__ __forceinline__ void trig64(float a, float& c, float& s) {
    double sd, cd;
    sincos((double)a, &sd, &cd);
    c = (float)cd; s = (float)sd;
}

__global__ void __launch_bounds__(128) compose_kernel(const ffb_entity* __restrict__ ents, int E, int B,
                                                      const float* __restrict__ sampled, int S, float* __restrict__ out_world) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    for (int e = 0; e < E; ++e) {
        const ffb_entity en = ents[e];
        M4 W;
#pragma unroll
        for (int k = 0; k < 16; ++k) W.m[k] = en.world[k];
        M4 local = W;
        if (en.randomizable) {
            float t[3] = {0.f, 0.f, 0.f}, r[3] = {0.f, 0.f, 0.f}, sc[3] = {1.f, 1.f, 1.f};
            const float* sb = sampled + (size_t)b * S * 3;
            if (en.s_translation >= 0) { t[0] = sb[en.s_translation * 3]; t[1] = sb[en.s_translation * 3 + 1]; t[2] = sb[en.s_translation * 3 + 2]; }
            if (en.s_rotation >= 0) { r[0] = sb[en.s_rotation * 3]; r[1] = sb[en.s_rotation * 3 + 1]; r[2] = sb[en.s_rotation * 3 + 2]; }
            if (en.s_scale >= 0) { sc[0] = sb[en.s_scale * 3]; sc[1] = sb[en.s_scale * 3 + 1]; sc[2] = sb[en.s_scale * 3 + 2]; }
            // entity/base.py:194-207: zMat = Pitch(r[2]) (about Y), yMat = Yaw(r[1]) (about Z), xMat = Roll(r[0]) (about X)
            float c, s;
            trig64(r[2], c, s);
            const float P[9] = {c, 0.f, s, 0.f, 1.f, 0.f, -s, 0.f, c};
            trig64(r[1], c, s);
            const float Y[9] = {c, -s, 0.f, s, c, 0.f, 0.f, 0.f, 1.f};
            trig64(r[0], c, s);
            const float R[9] = {1.f, 0.f, 0.f, 0.f, c, -s, 0.f, s, c};
            float PY[9], R3[9];
            mul3(P, Y, PY);
            mul3(PY, R, R3);
            M4 TC, R4;                       // (T + C): identity + translation, plus the centroid column
#pragma unroll
            for (int k = 0; k < 16; ++k) { TC.m[k] = 0.f; R4.m[k] = 0.f; }
            TC.m[0] = TC.m[5] = TC.m[10] = TC.m[15] = 1.f;
            TC.m[3] = t[0] + en.centroid[0]; TC.m[7] = t[1] + en.centroid[1]; TC.m[11] = t[2] + en.centroid[2];
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j) R4.m[i * 4 + j] = R3[i * 3 + j];
            R4.m[15] = 1.f;
            local = mul4(TC, R4);
            if (en.kind == FFB_ENTITY_MESH) {
                M4 Sm;
#pragma unroll
                for (int k = 0; k < 16; ++k) Sm.m[k] = 0.f;
                Sm.m[0] = sc[0]; Sm.m[5] = sc[1]; Sm.m[10] = sc[2]; Sm.m[15] = 1.f;
                local = mul4(local, Sm);
            }
            local = mul4(local, W);
        }
        float* o = out_world + ((size_t)b * E + e) * 16;
        if (en.parent >= e) {
            // a parent row that does not precede its child has no world matrix yet: fail loudly (NaN) instead of dropping the parent
#pragma unroll
            for (int k = 0; k < 16; ++k) local.m[k] = __int_as_float(0x7fc00000);
        } else if (en.parent >= 0) {
            M4 Pw;
            const float* pw = out_world + ((size_t)b * E + en.parent) * 16;
#pragma unroll
            for (int k = 0; k < 16; ++k) Pw.m[k] = pw[k];
            local = mul4(Pw, local);
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) o[k] = local.m[k];
    }
}

// ---- vertex transforms --------------------------------------------------------------------------------
constexpr int VT_THREADS = 256;
constexpr int VT_PER_THREAD = 4;                        // 4 vertices = 48 B = three 128-bit accesses
constexpr int VT_CHUNK = VT_THREADS * VT_PER_THREAD;

__device__ __forceinline__ void xform_point(const float* T, float x, float y, float z, float& ox, float& oy, float& oz) {
    // utils/math.py:220-228: T @ [x,y,z,1], then divide by w
    const float hx = fmaf(T[0], x, fmaf(T[1], y, fmaf(T[2], z, T[3])));
    const float hy = fmaf(T[4], x, fmaf(T[5], y, fmaf(T[6], z, T[7])));
    const float hz = fmaf(T[8], x, fmaf(T[9], y, fmaf(T[10], z, T[11])));
    const float hw = fmaf(T[12], x, fmaf(T[13], y, fmaf(T[14], z, T[15])));
    ox = hx / hw; oy = hy / hw; oz = hz / hw;
}
__device__ __forceinline__ void xform_dir(const float* T, float x, float y, float z, float& ox, float& oy, float& oz) {
    // utils/math.py:231-235: T @ [x,y,z,0], no divide
    ox = fmaf(T[0], x, fmaf(T[1], y, T[2] * z));
    oy = fmaf(T[4], x, fmaf(T[5], y, T[6] * z));
    oz = fmaf(T[8], x, fmaf(T[9], y, T[10] * z));
}

// 4 consecutive xyz vertices (48 B) at s: three 128-bit accesses when all four exist (n == 12 floats) and s is 16-byte
// aligned, scalar accesses otherwise (misaligned storage, tail); missing floats read as 0
__device__ __forceinline__ void ld_vert4(const float* __restrict__ s, int n, float v[12]) {
    if (n == 12 && ((reinterpret_cast<uintptr_t>(s) & 15) == 0)) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(s));
        const float4 b = __ldg(reinterpret_cast<const float4*>(s) + 1);
        const float4 c = __ldg(reinterpret_cast<const float4*>(s) + 2);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        v[8] = c.x; v[9] = c.y; v[10] = c.z; v[11] = c.w;
    } else {
#pragma unroll
        for (int k = 0; k < 12; ++k) v[k] = k < n ? __ldg(s + k) : 0.f;
    }
}
__device__ __forceinline__ void st_vert4(float* __restrict__ d, int n, const float v[12]) {
    if (n == 12 && ((reinterpret_cast<uintptr_t>(d) & 15) == 0)) {
        reinterpret_cast<float4*>(d)[0] = make_float4(v[0], v[1], v[2], v[3]);
        reinterpret_cast<float4*>(d)[1] = make_float4(v[4], v[5], v[6], v[7]);
        reinterpret_cast<float4*>(d)[2] = make_float4(v[8], v[9], v[10], v[11]);
    } else {
#pragma unroll
        for (int k = 0; k < 12; ++k)
            if (k < n) d[k] = v[k];
    }
}

template <bool DIRS>
__device__ __forceinline__ void xform_block4(const float* __restrict__ src, float* __restrict__ dst, long long v0, long long V,
                                             const float* T) {
    // src/dst point at vertex 0 of the mesh; this thread owns vertices [v0, v0+4)
    if (v0 >= V) return;
    const int n = v0 + 4 <= V ? 12 : (int)(V - v0) * 3;
    float in[12], o[12];
    ld_vert4(src + v0 * 3, n, in);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (DIRS) xform_dir(T, in[3 * k], in[3 * k + 1], in[3 * k + 2], o[3 * k], o[3 * k + 1], o[3 * k + 2]);
        else xform_point(T, in[3 * k], in[3 * k + 1], in[3 * k + 2], o[3 * k], o[3 * k + 1], o[3 * k + 2]);
    }
    st_vert4(dst + v0 * 3, n, o);
}

__global__ void __launch_bounds__(VT_THREADS) transform_vertices_kernel(const ffb_mesh_table mt, const float* __restrict__ verts,
                                                                        int E, const int32_t* __restrict__ anim_idx,
                                                                        const float* __restrict__ world, float* __restrict__ out) {
    __shared__ float T[16];
    const int b = blockIdx.y;
    // locate this CTA's mesh from the chunk prefix (M <= 32, uniform per CTA)
    int chunk = blockIdx.x, m = 0;
    for (; m < mt.M; ++m) {
        const int nch = (mt.voff[m + 1] - mt.voff[m] + VT_CHUNK - 1) / VT_CHUNK;
        if (chunk < nch) break;
        chunk -= nch;
    }
    if (m >= mt.M) return;
    if (threadIdx.x < 16) T[threadIdx.x] = world[((size_t)b * E + mt.entity[m]) * 16 + threadIdx.x];
    __syncthreads();
    const long long V = mt.voff[m + 1] - mt.voff[m];
    const long long vtot = mt.voff[mt.M];
    const float* src = verts + (size_t)mt.voff[m] * 3;
    if (mt.nframes[m] > 0 && mt.frames[m] != nullptr && anim_idx != nullptr) {
        int f = anim_idx[(size_t)b * mt.M + m];
        f = f < 0 ? 0 : (f >= mt.nframes[m] ? mt.nframes[m] - 1 : f);      // the reference would raise IndexError
        src = mt.frames[m] + (size_t)f * V * 3;
    }
    float* dst = out + ((size_t)b * vtot + mt.voff[m]) * 3;
    xform_block4<false>(src, dst, (long long)chunk * VT_CHUNK + threadIdx.x * VT_PER_THREAD, V, T);
}

template <bool DIRS>
__global__ void __launch_bounds__(VT_THREADS) transform_points_kernel(const float* __restrict__ pts, long long V,
                                                                      const float* __restrict__ Tg, float* __restrict__ out) {
    __shared__ float T[16];
    if (threadIdx.x < 16) T[threadIdx.x] = Tg[threadIdx.x];
    __syncthreads();
    xform_block4<DIRS>(pts, out, ((long long)blockIdx.x * VT_THREADS + threadIdx.x) * VT_PER_THREAD, V, T);
}

// backward of transform_points / transform_directions (utils/math.py:220-235, torch autograd of a broadcast matmul in the
// reference; the laser rays and the projector / camera matrices are optimised through it, projection/laser.py:262-275).
// Per point: y = h[:3] / h[3] with h = T @ [p, 1] (points) or y = (T @ [p, 0])[:3] (directions), d = dL/dh, then
//   d_pts[v] = (T^T d)[:3]            and            d_T[i][j] = sum_v d_i(v) p~_j(v),  p~ = (x, y, z, 1) or (x, y, z, 0).
// One template serves the points-only backward (DT off: one 4-vertex group per thread, 64-thread CTAs) and the
// matrix gradient (DT on: a grid-stride loop over at most TB_MAX_CTAS CTAs, fp32 sums per thread, an fp32 shuffle tree per
// warp, a fixed-order sum over the 8 warps, one 16-float partial per CTA).  The grid depends on V only -- not on the device
// -- so the summation order, and with it every bit of d_T, is the same on every call.
constexpr int TB_MAX_CTAS = 3 * kNumSMs;      // all resident at once: 3 CTAs x 256 threads per SM (<= 80 registers)
constexpr int TB_PTS_THREADS = 64;            // points only: small CTAs spread the V / 4 threads over every SM
constexpr int TB_FOLD_THREADS = 1024;

__host__ __device__ constexpr long long transform_bwd_grid(long long V, bool dT) {
    return dT ? ((V + VT_CHUNK - 1) / VT_CHUNK > TB_MAX_CTAS ? TB_MAX_CTAS : (V + VT_CHUNK - 1) / VT_CHUNK)
              : (V + TB_PTS_THREADS * VT_PER_THREAD - 1) / (TB_PTS_THREADS * VT_PER_THREAD);
}

template <bool DIRS>
__device__ __forceinline__ void xform_bwd_point(const float* T, float x, float y, float z, float g0, float g1, float g2, float d[4]) {
    if (DIRS) { d[0] = g0; d[1] = g1; d[2] = g2; d[3] = 0.f; }
    else {
        const float h0 = fmaf(T[0], x, fmaf(T[1], y, fmaf(T[2], z, T[3])));
        const float h1 = fmaf(T[4], x, fmaf(T[5], y, fmaf(T[6], z, T[7])));
        const float h2 = fmaf(T[8], x, fmaf(T[9], y, fmaf(T[10], z, T[11])));
        const float h3 = fmaf(T[12], x, fmaf(T[13], y, fmaf(T[14], z, T[15])));
        const float inv = 1.0f / h3;
        d[0] = g0 * inv; d[1] = g1 * inv; d[2] = g2 * inv;
        d[3] = -(g0 * h0 + g1 * h1 + g2 * h2) * inv * inv;
    }
}

// DT: `out` receives d_T itself when gridDim.x == 1, else this CTA's partial at out + 16 * blockIdx.x
template <bool DIRS, bool DPTS, bool DT, int THREADS = DT ? VT_THREADS : TB_PTS_THREADS>
__global__ void __launch_bounds__(THREADS, 3 * VT_THREADS / THREADS) transform_bwd_kernel(const float* __restrict__ pts, long long V,
                                                                      const float* __restrict__ Tg, const float* __restrict__ g,
                                                                      float* __restrict__ d_pts, float* __restrict__ out) {
    __shared__ float red[THREADS / 32][16];
    const float* T = Tg;                       // read where used: the loads overlap the first points' (no staging barrier)
    constexpr int R = DIRS ? 3 : 4;            // directions: row 3 and column 3 of d_T are zero
    float acc[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) acc[k] = 0.f;
    for (long long v0 = ((long long)blockIdx.x * THREADS + threadIdx.x) * VT_PER_THREAD; v0 < V;
         v0 += (long long)gridDim.x * THREADS * VT_PER_THREAD) {
        const int n = v0 + 4 <= V ? 12 : (int)(V - v0) * 3;
        float p[12], gi[12], o[12];
        ld_vert4(pts + v0 * 3, n, p);
        ld_vert4(g + v0 * 3, n, gi);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float x = p[3 * k], y = p[3 * k + 1], z = p[3 * k + 2];
            float d[4];
            xform_bwd_point<DIRS>(T, x, y, z, gi[3 * k], gi[3 * k + 1], gi[3 * k + 2], d);
            if (DPTS) {
                o[3 * k] = fmaf(T[0], d[0], fmaf(T[4], d[1], fmaf(T[8], d[2], T[12] * d[3])));
                o[3 * k + 1] = fmaf(T[1], d[0], fmaf(T[5], d[1], fmaf(T[9], d[2], T[13] * d[3])));
                o[3 * k + 2] = fmaf(T[2], d[0], fmaf(T[6], d[1], fmaf(T[10], d[2], T[14] * d[3])));
            }
            if (DT && 3 * k < n) {
#pragma unroll
                for (int i = 0; i < R; ++i) {
                    acc[4 * i] = fmaf(d[i], x, acc[4 * i]);
                    acc[4 * i + 1] = fmaf(d[i], y, acc[4 * i + 1]);
                    acc[4 * i + 2] = fmaf(d[i], z, acc[4 * i + 2]);
                    if (!DIRS) acc[4 * i + 3] += d[i];
                }
            }
        }
        if (DPTS) st_vert4(d_pts + v0 * 3, n, o);
    }
    if (!DT) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        if (k / 4 < R && (k % 4) < R) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], off);
        }
        if (lane == 0) red[warp][k] = acc[k];
    }
    __syncthreads();
    if (threadIdx.x < 16) {
        float s = red[0][threadIdx.x];
#pragma unroll
        for (int w = 1; w < THREADS / 32; ++w) s += red[w][threadIdx.x];
        out[(gridDim.x == 1 ? 0 : 16 * blockIdx.x) + threadIdx.x] = s;
    }
}

// d_T = sum of the G partials in fp64: 64 row groups sum every 64th partial in turn, then a fixed pairwise tree
__global__ void __launch_bounds__(TB_FOLD_THREADS) transform_bwd_fold_kernel(const float* __restrict__ partials, int G,
                                                                             float* __restrict__ d_T) {
    constexpr int ROWS = TB_FOLD_THREADS / 16;
    __shared__ double s[ROWS][16];
    const int j = threadIdx.x & 15, r = threadIdx.x >> 4;
    double a = 0.0;
    for (int c = r; c < G; c += ROWS) a += (double)partials[16 * c + j];
    s[r][j] = a;
    __syncthreads();
#pragma unroll
    for (int h = ROWS / 2; h > 0; h >>= 1) {
        if (r < h) s[r][j] += s[r + h][j];
        __syncthreads();
    }
    if (threadIdx.x < 16) d_T[threadIdx.x] = (float)s[0][threadIdx.x];
}

template <bool DPTS, bool DT>
static void launch_transform_bwd(bool dirs, unsigned grid, const float* pts, long long V, const float* T, const float* g,
                                 float* d_pts, float* out, cudaStream_t st) {
    constexpr int threads = DT ? VT_THREADS : TB_PTS_THREADS;
    if (dirs) transform_bwd_kernel<true, DPTS, DT><<<grid, threads, 0, st>>>(pts, V, T, g, d_pts, out);
    else transform_bwd_kernel<false, DPTS, DT><<<grid, threads, 0, st>>>(pts, V, T, g, d_pts, out);
}

__global__ void __launch_bounds__(128) clamp_fov_kernel(const float* __restrict__ rays, int N, const float* __restrict__ M,
                                                        const float* __restrict__ Minv, float lo, float hi, float* __restrict__ out) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float Tm[16], Ti[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) { Tm[k] = M[k]; Ti[k] = Minv[k]; }
    float x, y, z;
    xform_point(Tm, rays[3 * n], rays[3 * n + 1], rays[3 * n + 2], x, y, z);    // projectRaysToNDC
    x = fminf(fmaxf(x, lo), hi);                                                   // torch.clamp(ndc[:,0:2], 1-c, c)
    y = fminf(fmaxf(y, lo), hi);
    float wx, wy, wz;
    xform_point(Ti, x, y, z, wx, wy, wz);                                          // projectNDCPointsToWorld
    const float nrm = sqrtf(wx * wx + wy * wy + wz * wz);                          // laser.normalize
    out[3 * n] = wx / nrm; out[3 * n + 1] = wy / nrm; out[3 * n + 2] = wz / nrm;
}

// Laser.randomize_laser_out_of_bounds / randomize_camera_out_of_bounds (projection/laser.py:208-249) in one launch, no host
// sync: a ray whose NDC x or y lies outside (lo, hi) is respawned at (u0, u1, -1) un-projected through Minv; if ANY ray was
// out of bounds all rays are renormalised, otherwise nothing is written (the reference returns before its normalise).
// One CTA walks all rays: count and exclusive scan of the out-of-bounds flags give the k-th respawned ray row k of the
// injected variates (the reference draws torch.rand(K, 3) for the K rays in index order); the Philox mode keys by ray.
constexpr int RS_THREADS = 1024;
__global__ void __launch_bounds__(RS_THREADS) respawn_kernel(float* __restrict__ rays, int N, const float* __restrict__ M,
                                                             const float* __restrict__ ndc_in, float lo, float hi,
                                                             const float* __restrict__ Minv, uint64_t seed, uint64_t counter,
                                                             const float* __restrict__ variates, int* __restrict__ count_out) {
    __shared__ int warp_cnt[32];
    __shared__ int carry;
    __shared__ float Tm[16], Ti[16];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid < 16) { Tm[tid] = M ? M[tid] : 0.f; Ti[tid] = Minv[tid]; }
    if (tid == 0) carry = 0;
    __syncthreads();
    // pass 1: is anything out of bounds?
    int mine = 0;
    for (int n = tid; n < N; n += RS_THREADS) {
        float x, y, z;
        if (M) xform_point(Tm, rays[3 * n], rays[3 * n + 1], rays[3 * n + 2], x, y, z);
        else { x = ndc_in[3 * n]; y = ndc_in[3 * n + 1]; }
        mine += (x >= hi || x <= lo || y >= hi || y <= lo) ? 1 : 0;
    }
    const int any = __syncthreads_count(mine);
    if (any == 0) {
        if (tid == 0 && count_out) *count_out = 0;
        return;
    }
    // pass 2: respawn in index order, renormalise everything
    for (int base = 0; base < N; base += RS_THREADS) {
        const int n = base + tid;
        bool oob = false;
        float rx = 0.f, ry = 0.f, rz = 0.f;
        if (n < N) {
            rx = rays[3 * n]; ry = rays[3 * n + 1]; rz = rays[3 * n + 2];
            float x, y, z;
            if (M) xform_point(Tm, rx, ry, rz, x, y, z);
            else { x = ndc_in[3 * n]; y = ndc_in[3 * n + 1]; }
            oob = x >= hi || x <= lo || y >= hi || y <= lo;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, oob);
        if (lane == 0) warp_cnt[w] = __popc(bal);
        __syncthreads();
        int before = carry;
        for (int k = 0; k < w; ++k) before += warp_cnt[k];
        const int row = before + __popc(bal & ((1u << lane) - 1u));
        if (oob) {
            float u0, u1;
            if (variates) { u0 = variates[3 * row]; u1 = variates[3 * row + 1]; }
            else {
                uint32_t r[4];
                Philox::gen(seed, (uint32_t)n, (uint32_t)counter, (uint32_t)(counter >> 32), 0x52455350u, r);
                u0 = Philox::u01(r[0]); u1 = Philox::u01(r[1]);
            }
            xform_point(Ti, u0, u1, -1.0f, rx, ry, rz);
        }
        if (n < N) {
            const float nrm = sqrtf(rx * rx + ry * ry + rz * rz);
            rays[3 * n] = rx / nrm; rays[3 * n + 1] = ry / nrm; rays[3 * n + 2] = rz / nrm;
        }
        __syncthreads();
        if (tid == 0) {
            int t = 0;
            for (int k = 0; k < RS_THREADS / 32; ++k) t += warp_cnt[k];
            carry += t;
        }
        __syncthreads();
    }
    if (tid == 0 && count_out) *count_out = carry;
}

}  // namespace scene
}  // namespace ffb

using namespace ffb;
using namespace ffb::scene;

extern "C" int ffb_respawn_rays(float* rays, int32_t N, const float* M, const float* ndc, float lo, float hi, const float* Minv,
                                uint64_t seed, uint64_t counter, const float* variates, int32_t* respawned_out, void* stream) {
    if (!rays || !Minv || N <= 0) return fail_arg(FFB_E_ARG, "respawn_rays: bad argument");
    if ((M == nullptr) == (ndc == nullptr)) return fail_arg(FFB_E_ARG, "respawn_rays: exactly one of M (project the rays) and ndc (given coordinates) is required");
    respawn_kernel<<<1, RS_THREADS, 0, as_stream(stream)>>>(rays, N, M, ndc, lo, hi, Minv, seed, counter, variates, respawned_out);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_sample(ffb_sampler* samplers, int32_t S, int32_t B, int32_t mode, uint64_t seed, uint64_t sample0,
                          const float* variates, float* out, void* stream) {
    if (!samplers || !out || S <= 0 || B <= 0) return fail_arg(FFB_E_ARG, "sample: bad argument");
    if (mode == FFB_MODE_INJECTED && !variates) return fail_arg(FFB_E_ARG, "sample: injected mode needs variates");
    if (mode != FFB_MODE_TRAIN && mode != FFB_MODE_EVAL && mode != FFB_MODE_INJECTED) return fail_arg(FFB_E_ARG, "sample: unknown mode");
    cudaStream_t st = as_stream(stream);
    if (mode == FFB_MODE_EVAL) sample_eval_kernel<<<(S + 127) / 128, 128, 0, st>>>(samplers, S, B, out);
    else sample_kernel<<<(unsigned)(((long long)B * S + 255) / 256), 256, 0, st>>>(samplers, S, B, mode, seed, sample0, variates, out);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_uniform_between(const float* a, const float* b, const float* u, int64_t n, float* out, void* stream) {
    if (!a || !b || !u || !out || n < 0) return fail_arg(FFB_E_ARG, "uniform_between: bad argument");
    if (n == 0) return 0;
    uniform_between_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(a, b, u, n, out);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_sample_anim_index(const int32_t* amin, const int32_t* amax, int32_t* cur, int32_t M, int32_t B, int32_t mode,
                                     uint64_t seed, uint64_t sample0, int32_t* out, void* stream) {
    if (!amin || !amax || !out || M <= 0 || B <= 0) return fail_arg(FFB_E_ARG, "sample_anim_index: bad argument");
    if (mode == FFB_MODE_EVAL && !cur) return fail_arg(FFB_E_ARG, "sample_anim_index: eval mode needs the cursor array");
    if (mode != FFB_MODE_TRAIN && mode != FFB_MODE_EVAL) return fail_arg(FFB_E_ARG, "sample_anim_index: mode must be train or eval");
    const long long n = mode == FFB_MODE_EVAL ? M : (long long)B * M;
    anim_index_kernel<<<(unsigned)((n + 127) / 128), 128, 0, as_stream(stream)>>>(amin, amax, cur, M, B, mode, seed, sample0, out);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_compose_world(const ffb_entity* entities, int32_t E, int32_t B, const float* sampled, int32_t S,
                                 float* out_world, void* stream) {
    if (!entities || !out_world || E <= 0 || B <= 0) return fail_arg(FFB_E_ARG, "compose_world: bad argument");
    if (S > 0 && !sampled) return fail_arg(FFB_E_ARG, "compose_world: null sampled");
    compose_kernel<<<(B + 127) / 128, 128, 0, as_stream(stream)>>>(entities, E, B, sampled, S, out_world);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_transform_vertices(const ffb_mesh_table* meshes, const float* verts, int32_t E, int32_t B,
                                      const int32_t* anim_idx, const float* world, float* out, void* stream) {
    if (!meshes || !world || !out || E <= 0 || B <= 0) return fail_arg(FFB_E_ARG, "transform_vertices: bad argument");
    if (meshes->M <= 0 || meshes->M > FFB_MAX_MESHES) return fail_arg(FFB_E_LIMIT, "transform_vertices: M must be in [1, FFB_MAX_MESHES]");
    if (B > 65535) return fail_arg(FFB_E_LIMIT, "transform_vertices: B > 65535");
    long long chunks = 0;
    for (int m = 0; m < meshes->M; ++m) {
        const int v = meshes->voff[m + 1] - meshes->voff[m];
        if (v < 0) return fail_arg(FFB_E_ARG, "transform_vertices: voff must be non-decreasing");
        if (meshes->entity[m] < 0 || meshes->entity[m] >= E) return fail_arg(FFB_E_ARG, "transform_vertices: entity row out of range");
        if (!(meshes->nframes[m] > 0 && meshes->frames[m]) && !verts) return fail_arg(FFB_E_ARG, "transform_vertices: null verts");
        chunks += (v + VT_CHUNK - 1) / VT_CHUNK;
    }
    if (chunks == 0) return 0;
    transform_vertices_kernel<<<dim3((unsigned)chunks, B), VT_THREADS, 0, as_stream(stream)>>>(*meshes, verts, E, anim_idx, world, out);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_transform_points(const float* pts, int64_t V, const float* T, int as_directions, float* out, void* stream) {
    if (!pts || !T || !out || V < 0) return fail_arg(FFB_E_ARG, "transform_points: bad argument");
    if (V == 0) return 0;
    const unsigned grid = (unsigned)((V + VT_CHUNK - 1) / VT_CHUNK);
    if (as_directions) transform_points_kernel<true><<<grid, VT_THREADS, 0, as_stream(stream)>>>(pts, V, T, out);
    else transform_points_kernel<false><<<grid, VT_THREADS, 0, as_stream(stream)>>>(pts, V, T, out);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_transform_points_bwd(const float* pts, int64_t V, const float* T, int as_directions, const float* g_out,
                                        float* d_pts, void* stream) {
    if (!pts || !T || !g_out || !d_pts || V < 0) return fail_arg(FFB_E_ARG, "transform_points_bwd: bad argument");
    if (V == 0) return 0;
    launch_transform_bwd<true, false>(as_directions, (unsigned)transform_bwd_grid(V, false), pts, V, T, g_out, d_pts, nullptr,
                                      as_stream(stream));
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" size_t ffb_transform_bwd_workspace_bytes(int64_t V) {
    if (V < 0) { fail_arg(FFB_E_ARG, "transform_bwd_workspace_bytes: V < 0"); return 0; }
    const long long G = transform_bwd_grid(V, true);
    return G > 1 ? (size_t)G * 16 * sizeof(float) : 0;
}

extern "C" int ffb_transform_points_bwd_full(const float* pts, int64_t V, const float* T, int as_directions, const float* g_out,
                                             float* d_pts, float* d_T, void* workspace, size_t workspace_bytes, void* stream) {
    if (!pts || !T || !g_out || !d_T || V < 0) return fail_arg(FFB_E_ARG, "transform_points_bwd_full: bad argument");
    const size_t need = ffb_transform_bwd_workspace_bytes(V);
    if (need && !workspace) return fail_arg(FFB_E_ARG, "transform_points_bwd_full: null workspace");
    if (workspace_bytes < need) return fail_arg(FFB_E_WORKSPACE, "transform_points_bwd_full: workspace too small");
    const cudaStream_t st = as_stream(stream);
    if (V == 0) {
        FFB_CUDA(cudaMemsetAsync(d_T, 0, 16 * sizeof(float), st));
        return 0;
    }
    const int G = (int)transform_bwd_grid(V, true);
    float* out = G > 1 ? static_cast<float*>(workspace) : d_T;
    if (d_pts) launch_transform_bwd<true, true>(as_directions, G, pts, V, T, g_out, d_pts, out, st);
    else launch_transform_bwd<false, true>(as_directions, G, pts, V, T, g_out, nullptr, out, st);
    FFB_CUDA(cudaGetLastError());
    if (G > 1) {
        transform_bwd_fold_kernel<<<1, TB_FOLD_THREADS, 0, st>>>(out, G, d_T);
        FFB_CUDA(cudaGetLastError());
    }
    return 0;
}

extern "C" int ffb_rays_to_ndc(const float* rays, int32_t N, const float* M, float* ndc, void* stream) {
    return ffb_transform_points(rays, N, M, 0, ndc, stream);
}

extern "C" int ffb_clamp_to_fov(const float* rays, int32_t N, const float* M, const float* Minv, float clamp_lo, float clamp_hi,
                                float* rays_out, void* stream) {
    if (!rays || !M || !Minv || !rays_out || N <= 0) return fail_arg(FFB_E_ARG, "clamp_to_fov: bad argument");
    clamp_fov_kernel<<<(N + 127) / 128, 128, 0, as_stream(stream)>>>(rays, N, M, Minv, clamp_lo, clamp_hi, rays_out);
    FFB_CUDA(cudaGetLastError());
    return 0;
}
