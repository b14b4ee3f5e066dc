// Warp-tile splat kernels (included by ffb_splat.cu inside namespace ffb::splat).
//
// What the ncu captures of the earlier CTA-tile kernels showed (profiles/r01a_baseline): DRAM traffic equals the
// algorithmic bytes, but only ~22 % of the issued instructions were splat arithmetic -- the rest was per-CTA staging,
// three block barriers per candidate chunk (29 % of the stall samples) and per-lane culling -- and half of the
// evaluated (texel, point) pairs lay outside the point's window (8x32 warp blocks around a 43x43 footprint).
//
// This version removes the CTA from the picture:
//   * the binning kernel builds one candidate list per 64x16 SUPER TILE; a list entry is the 32-byte record the
//     kernel needs (scaled position, window origin, row / column span, point index) -- no index indirection, no
//     in-kernel culling;
//   * a warp owns a strip of four vertically adjacent super tiles from the first load to the last store: no
//     __syncthreads, only __syncwarp around a small per-warp shared table.  The strip's list offsets are fetched with
//     one load, and the candidate records (and, in the backward, the upstream gradients) of the next super tile are
//     in flight while the current one is computed -- the two dependent global loads at the head of a warp's life
//     were a quarter of all stall samples before.  Per super tile it stages the candidates once and then walks the
//     four 16x16 tiles; the 16 rows are common to all four, so everything that depends on (candidate, row) only -- (r - P1)^2,
//     r - P1, the row masks -- is computed once per warp and read back with one LDS.128 per group;
//   * inside a 16x16 tile lane = (column 0..15, row half 0..1); the packed fp32 pipe (FADD2/FMUL2/FFMA2) handles
//     two rows per lane, so one warp instruction covers a 16x4 texel group.  Tiles outside a candidate's column
//     span are skipped through warp-uniform ballot masks; all four row groups of a touched tile are evaluated
//     (branch-free, four independent dependency chains per lane): 3364 evaluated pairs per point for a 43x43 window
//     instead of 3700, at a third of the instructions;
//   * the column mask of the sum window is a lane predicate on the accumulate, so masks cost no arithmetic;
//   * g = 2^(d2^2 * K), K = -log2(e)/sigma^2, with d2 = dc*dc + dr*dr rounded exactly like the reference: the inner
//     group is LDS.128 + FADD2 + 2 FMUL2 + 2 MUFU.EX2 + 2 FFMA2.  With 16 MUFU lanes per SM the exp is the busiest
//     pipe, which is why the evaluated-pair count above matters;
//   * soft-OR needs no window at all when the footprint is at least the exact no-op radius (g <= 2^-25 rounds 1-g
//     to 1): texels outside contribute a bit-exact factor of 1;
//   * backward: with the forward's soft-OR output at hand (saved_softor) the per-texel product is 1 - O and a single
//     pass suffices; otherwise a first pass rebuilds it.  Per-lane d/dP partial sums are parked in shared memory
//     across the four tiles, then folded across the warp with five shuffles for both components at once and leave
//     the warp as one atomic per component per (candidate, super tile);
//   * super tiles with more than 16 candidates (clustered patterns) are left to the overflow kernels at the end of
//     this file, which walk the binning kernel's overflow list with the same device functions in chunks of 16.
#pragma once

constexpr int WT_S = 1;                   // vertically adjacent super tiles per warp (<= 16: one lane pair per super tile holds its list bounds).  Backward:
                                          // 0.624 / 0.658 / 0.654 / 0.651 ms per 64 samples at 1 / 2 / 3 / 4 (locality of the CTAs in flight beats the
                                          // cross-super-tile prefetch a longer strip allows)
constexpr int WF_S = 1;                   // ... in the TMA-store forward.  Measured per 64 samples (256-thread CTAs): 0.422 / 0.419 / 0.475 / 0.541 /
                                          // 0.587 ms at 1 / 2 / 4 / 8 / 16: with short strips the CTAs in flight (scheduled column block first) write a
                                          // narrow band of texture rows at any time, and DRAM sees whole rows complete together
constexpr int WT_CTA = 256;               // forward / overflow kernels: 8 warps x 4 super tiles (64 x 16 texels each) = 64 x 512 texels
constexpr int WT_WARPS = WT_CTA / 32;
constexpr int WF_CTA = 64;                // TMA-store forward (measured at one super tile per warp: 0.386 / 0.379 / 0.378 ms at 128 / 64 / 32 threads)
constexpr int WF_WARPS = WF_CTA / 32;
constexpr int WF_MINB = 1024 / WF_CTA;    // 32 warps per SM at 64 registers
constexpr int WB_CTA = 32;                // backward: one warp per CTA (measured 0.67 ms vs 0.70 ms at 64 / 128 threads: a strip's slot frees the moment it ends; the forward prefers 8 warps)
constexpr int WB_WARPS = WB_CTA / 32;
constexpr int FWD_MINB = 4;               // resident CTAs per SM the register allocation aims for
constexpr int BWD_MINB = 22;              // 22-24 warps per SM: what 80 registers and ~10 KB of shared memory per warp allow

constexpr int TMA_TILE_BYTES = WT * WT * 4;   // one 16x16 fp32 tile as a TMA box

struct WtConsts {
    float K2;                             // -log2(e) / sigma^2
    float thr_s, thr_o;                   // 4*H + 2 for the sum / soft-OR row masks
    float hs, ho;                         // H + 0.5 for the column predicates
    float c1;                             // 1 + 2^-23: keeps 1 - g away from 0 in the backward quotient
    float disc2;                          // squared radius beyond which g < 1e-7 (backward tile culling; wt_consts)
    float disc2_f;                        // squared radius beyond which g <= 2^-25 (forward tile culling: 1 - g == 1 exactly)
    float near2;                          // squared radius beyond which g < 2^-8 (backward: far tiles need no reciprocal)
    float s2, rs2;                        // sqrt(-K2) and its reciprocal: the backward's tables hold d^2 * s2, so g = 2^-(d2s^2)
    // super-tile backward (ffb_splat_st.cuh): distances themselves are scaled by r1 = sqrt(s2)
    float r1, rs3;                        // r1 and 1 / (s2 * r1), which undoes the scaling of g * d2s * dxs
    float hs_r;                           // (H_s + 0.5) * r1: row predicate of the sum window on scaled offsets
    float m_r, thr_r;                     // column mask of the sum window: saturate(thr_r + m_r * |e * r1|), m_r = -4 / r1, thr_r = 4 H_s + 2
};

__device__ __forceinline__ float ex2_approx(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// volatile twins: ptxas keeps volatile asm statements in source order, which is how the staged backward loop pins
// "all exponentials, then all reciprocals"
__device__ __forceinline__ float ex2_approx_v(float x) {
    float r;
    asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float rcp_approx_v(float x) {
    float r;
    asm volatile("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float cheb_mask(float e, float thr) {      // 1 if |e| <= H else 0 (e integer valued)
    return __saturatef(fmaf(fabsf(e), -4.f, thr));
}
__device__ __forceinline__ float2 bc(float x) { return make_float2(x, x); }
__device__ __forceinline__ float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }

// Per-warp staging: candidate records and the (candidate, row pair) tables of the warp's 16 rows.
// TABB: 0 = no second table, 1 = dy only (float2), 2 = dy + soft-OR row mask (float4).  ACC: backward partial-sum parking.
// TIN: backward staging buffers for the upstream tile (cp.async targets).  NRAW: record buffers (2 = double buffered).
template <int TABB, bool ACC = false, bool TIN = false, int NRAW = 2>
struct WarpStage {
    float4 cand[WCH];                     // p0, f0, point index (bits), row-group mask (bits)
    float2 prow[WCH];                     // p1, f1
    float4 tabA[WCH][WT / 2];             // dy^2 (2 rows), sum row mask (2 rows)
    float4 tabB4[TABB == 2 ? WCH : 1][WT / 2];   // dy (2 rows), soft-OR row mask (2 rows)
    float2 tabB2[TABB == 1 ? WCH : 1][WT / 2];   // dy (2 rows)
    uint4 raw[NRAW][2 * WCH];             // candidate records as fetched by cp.async
    float acc[ACC ? WCH : 1][33];   // backward: parked d/dP partial sums (first half: d/dp0, second: d/dp1), row padded
    float tin[TIN ? 2 : 1][TIN ? WT : 1][TIN ? 24 : 4];   // backward: upstream soft-OR gradient / saved output tile, rows padded to 24 (bank-conflict free)
};

// Which staged candidates touch which 16x16 tile: warp-uniform ballots, 16 bits per tile.
struct WtMasks {
    unsigned tb01, tb23;                  // touched (and, in the backward, inside the culling disc)
    unsigned nb01, nb23;                  // backward: near tiles (some g >= 2^-8)
};
__device__ __forceinline__ unsigned tile_mask(const WtMasks& mk, int j) {
    return (((j & 2) ? mk.tb23 : mk.tb01) >> (16 * (j & 1))) & 0xffffu;
}
__device__ __forceinline__ unsigned near_mask(const WtMasks& mk, int j) {
    return (((j & 2) ? mk.nb23 : mk.nb01) >> (16 * (j & 1))) & 0xffffu;
}

// a lane's candidate record, as loaded (lane k holds candidate k of the chunk)
struct EntryRegs {
    float4 a;                             // p0, p1, f0, f1
    uint4 b;                              // row span, column span, point index, -
};
__device__ __forceinline__ EntryRegs load_entry(const Entry* __restrict__ entries, int base, int n, int lane) {
    EntryRegs e;
    e.a = make_float4(0.f, 0.f, 0.f, 0.f);
    e.b = make_uint4(0u, 0u, 0u, 0u);
    if (lane < n) {
        e.a = __ldg(reinterpret_cast<const float4*>(entries + base + lane));
        e.b = __ldg(reinterpret_cast<const uint4*>(entries + base + lane) + 1);
    }
    return e;
}

// asynchronous copy of n (<= WCH) records into a raw buffer: no registers held while the data is in flight
__device__ __forceinline__ void prefetch_entries(uint4* raw, const Entry* __restrict__ src, int n, int lane) {
    if (lane < 2 * n) {
        const unsigned dst = (unsigned)__cvta_generic_to_shared(raw + lane);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(reinterpret_cast<const uint4*>(src) + lane) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}
__device__ __forceinline__ EntryRegs take_entry(const uint4* raw, int n, int lane) {
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    EntryRegs e;
    e.a = make_float4(0.f, 0.f, 0.f, 0.f);
    e.b = make_uint4(0u, 0u, 0u, 0u);
    if (lane < n) {
        const uint4 a = raw[2 * lane];
        e.a = make_float4(__uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(a.z), __uint_as_float(a.w));
        e.b = raw[2 * lane + 1];
    }
    return e;
}

template <typename Stage>
struct StageTraits;
template <int TABB, bool ACC, bool TIN, int NRAW>
struct StageTraits<WarpStage<TABB, ACC, TIN, NRAW>> {
    static constexpr int tabb = TABB;
    static constexpr bool acc = ACC;
};

template <typename Stage>
__device__ __forceinline__ WtMasks stage_regs(Stage& s, const EntryRegs& e, int n, int c0, const float r0f,
                                              const WtConsts& fc, int lane) {
    constexpr int TABB = StageTraits<Stage>::tabb;
    constexpr bool ACC = StageTraits<Stage>::acc;
    __syncwarp();                         // previous chunk fully consumed
    bool ta[4] = {false, false, false, false};
    bool na[4] = {false, false, false, false};
    if (lane < n) {
        const int clo = (int)(e.b.y & 0xffff) - c0, chi = (int)(e.b.y >> 16) - c0;  // spans relative to the super tile
        const int r0 = (int)r0f, rlo = (int)(e.b.x & 0xffff) - r0, rhi = (int)(e.b.x >> 16) - r0;
        unsigned gm = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            ta[i] = clo < WT * i + WT && chi > WT * i;
            if (rlo < 4 * i + 4 && rhi > 4 * i) gm |= 1u << i;
        }
        // backward: a tile whose nearest texel centre has g < 1e-7 contributes nothing measurable to d/dP (weights
        // g * d2 * (c - P)); corner tiles of the square window go.  Forward: the radius is where g <= 2^-25, i.e. where
        // the soft-OR factor 1 - g is exactly 1 and a sum term is below 3e-8 (half an ulp of a texel value of 0.5; the
        // reference's own dense and baked sums differ by 2.4e-7).
        const float ry = fmaxf(fmaxf(r0f - e.a.y, e.a.y - (r0f + (float)(WT - 1))), 0.f);
        const float ry2 = ry * ry;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float xl = (float)(c0 + WT * i);
            const float rx = fmaxf(fmaxf(xl - e.a.x, e.a.x - (xl + (float)(WT - 1))), 0.f);
            const float rr = fmaf(rx, rx, ry2);
            ta[i] = ta[i] && rr <= (ACC ? fc.disc2 : fc.disc2_f);
            na[i] = ta[i] && rr < fc.near2;
        }
        s.cand[lane] = make_float4(e.a.x, e.a.z, __uint_as_float(e.b.z), __uint_as_float(gm));
        s.prow[lane] = make_float2(e.a.y, e.a.w);
    }
    if (ACC)
        for (int k = 0; k < n; ++k) s.acc[k][lane] = 0.f;
    WtMasks m;
    m.tb01 = __ballot_sync(0xffffffffu, ta[0]) | (__ballot_sync(0xffffffffu, ta[1]) << 16);
    m.tb23 = __ballot_sync(0xffffffffu, ta[2]) | (__ballot_sync(0xffffffffu, ta[3]) << 16);
    m.nb01 = m.tb01; m.nb23 = m.tb23;
    if (ACC) {
        m.nb01 = __ballot_sync(0xffffffffu, na[0]) | (__ballot_sync(0xffffffffu, na[1]) << 16);
        m.nb23 = __ballot_sync(0xffffffffu, na[2]) | (__ballot_sync(0xffffffffu, na[3]) << 16);
    }
    __syncwarp();
    const float rp = r0f + (float)(2 * (lane & 7));
    for (int t = lane; t < n * (WT / 2); t += 32) {
        const int k = t >> 3, p = t & 7;
        const float2 pf = s.prow[k];
        const float ra = rp, rb = rp + 1.f;
        const float da = ra - pf.x, db = rb - pf.x;
        const float ea = ra - pf.y, eb = rb - pf.y;
        // backward (ACC): squared distances pre-scaled by s2 = sqrt(-K2), so that g = 2^-(d2s * d2s) needs no multiply by K2
        const float sc = ACC ? fc.s2 : 1.f;
        s.tabA[k][p] = make_float4(__fmul_rn(da, da) * sc, __fmul_rn(db, db) * sc, cheb_mask(ea, fc.thr_s), cheb_mask(eb, fc.thr_s));
        if (TABB == 2) s.tabB4[k][p] = make_float4(da, db, cheb_mask(ea, fc.thr_o), cheb_mask(eb, fc.thr_o));
        if (TABB == 1) s.tabB2[k][p] = make_float2(da, db);
    }
    __syncwarp();
    return m;
}

// rows held by lane (c, h): 4i + 2h + {0,1}, i = 0..3  <->  one contiguous run of 8 rows (8h .. 8h+7) for the
// transposed ([ts0, ts1]) layout.  v[2i + j] in, w[0..7] = rows 8h..8h+7 out (and back).
__device__ __forceinline__ void rows_to_run(const float (&v)[8], float (&w)[8], int h) {
    float snd[4], rcv[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) snd[k] = h ? v[k] : v[4 + k];
#pragma unroll
    for (int k = 0; k < 4; ++k) rcv[k] = __shfl_xor_sync(0xffffffffu, snd[k], 16);
    // h = 0 keeps its groups 0,1 (rows 0,1,4,5) and receives the partner's groups 0,1 (rows 2,3,6,7);
    // h = 1 keeps its groups 2,3 (rows 10,11,14,15) and receives the partner's groups 2,3 (rows 8,9,12,13)
    if (h == 0) { w[0] = v[0]; w[1] = v[1]; w[2] = rcv[0]; w[3] = rcv[1]; w[4] = v[2]; w[5] = v[3]; w[6] = rcv[2]; w[7] = rcv[3]; }
    else        { w[0] = rcv[0]; w[1] = rcv[1]; w[2] = v[4]; w[3] = v[5]; w[4] = rcv[2]; w[5] = rcv[3]; w[6] = v[6]; w[7] = v[7]; }
}
__device__ __forceinline__ void run_to_rows(const float (&w)[8], float (&v)[8], int h) {
    float snd[4], rcv[4];
    // h = 0 holds rows 0..7: rows 2,3,6,7 belong to the partner; h = 1 holds rows 8..15: rows 8,9,12,13 belong to the partner
    if (h == 0) { snd[0] = w[2]; snd[1] = w[3]; snd[2] = w[6]; snd[3] = w[7]; }
    else        { snd[0] = w[0]; snd[1] = w[1]; snd[2] = w[4]; snd[3] = w[5]; }
#pragma unroll
    for (int k = 0; k < 4; ++k) rcv[k] = __shfl_xor_sync(0xffffffffu, snd[k], 16);
    if (h == 0) { v[0] = w[0]; v[1] = w[1]; v[2] = w[4]; v[3] = w[5]; v[4] = rcv[0]; v[5] = rcv[1]; v[6] = rcv[2]; v[7] = rcv[3]; }
    else        { v[0] = rcv[0]; v[1] = rcv[1]; v[2] = rcv[2]; v[3] = rcv[3]; v[4] = w[2]; v[5] = w[3]; v[6] = w[6]; v[7] = w[7]; }
}

// Position of a lane inside the super tile whose first texel is (r0, c0) of sample b.
struct WtCoord {
    int b, c0, r0, h, lc;
};

// Tile access.  A lane addresses its first texel once per super tile (TilePtr) and then steps from tile to tile;
// natural [ts1, ts0]: v[2i + j] <-> row r0 + 4i + 2h + j, column c;  transposed [ts0, ts1] (baked_sum_2's
// orientation): the lane moves rows 8h..8h+7 of its column as 2 x 128 bit.
struct TilePtr {
    size_t nat;        // element offset of (row r0 + 2h, column c0 + lc) in a natural frame of sample b
    size_t tr;         // element offset of (column c0 + lc, row r0 + 8h) in a transposed frame of sample b
};
__device__ __forceinline__ TilePtr tile_ptr(const RasterParams& q, const WtCoord& w) {
    TilePtr t;
    t.nat = ((size_t)w.b * q.ts1 + (w.r0 + 2 * w.h)) * q.ts0 + w.c0 + w.lc;
    t.tr = ((size_t)w.b * q.ts0 + w.c0 + w.lc) * q.ts1 + w.r0 + 8 * w.h;
    return t;
}

__device__ __forceinline__ void store_natural(float* __restrict__ o, const RasterParams& q, const WtCoord& w, int c, bool interior,
                                              const float (&v)[8]) {
    if (interior) {                                        // warp-uniform
        float* r = o;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            r[0] = v[2 * i];
            r[q.ts0] = v[2 * i + 1];
            r += 4 * (size_t)q.ts0;
        }
    } else if (c < q.ts0) {
        const int rb = w.r0 + 2 * w.h;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j)
                if (rb + 4 * i + j < q.ts1) o[(size_t)(4 * i + j) * q.ts0] = v[2 * i + j];
    }
}
__device__ __forceinline__ void load_natural(const float* __restrict__ p, const RasterParams& q, const WtCoord& w, int c, bool interior,
                                             float (&v)[8]) {
    if (interior) {
        const float* r = p;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            v[2 * i] = __ldg(r);
            v[2 * i + 1] = __ldg(r + q.ts0);
            r += 4 * (size_t)q.ts0;
        }
    } else {
        const int rb = w.r0 + 2 * w.h;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j)
                v[2 * i + j] = (c < q.ts0 && rb + 4 * i + j < q.ts1) ? __ldg(p + (size_t)(4 * i + j) * q.ts0) : 0.f;
    }
}
__device__ __forceinline__ void store_run(float* __restrict__ o, const RasterParams& q, const WtCoord& w, int c, bool interior,
                                          const float (&run)[8]) {
    if (interior && (q.ts1 & 7) == 0) {                     // one 256-bit store: a full 32-byte sector per lane
        asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(o), "f"(run[0]), "f"(run[1]), "f"(run[2]),
                     "f"(run[3]), "f"(run[4]), "f"(run[5]), "f"(run[6]), "f"(run[7]) : "memory");
    } else if (c < q.ts0) {
        const int rr = w.r0 + 8 * w.h;
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (rr + k < q.ts1) o[k] = run[k];
    }
}
__device__ __forceinline__ void load_run(const float* __restrict__ p, const RasterParams& q, const WtCoord& w, int c, bool interior,
                                         float (&run)[8]) {
    if (interior && (q.ts1 & 7) == 0) {                     // one 256-bit load: a full 32-byte sector per lane
        asm volatile("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];" : "=f"(run[0]), "=f"(run[1]), "=f"(run[2]),
                     "=f"(run[3]), "=f"(run[4]), "=f"(run[5]), "=f"(run[6]), "=f"(run[7]) : "l"(p));
    } else {
        const int rr = w.r0 + 8 * w.h;
#pragma unroll
        for (int k = 0; k < 8; ++k) run[k] = (c < q.ts0 && rr + k < q.ts1) ? __ldg(p + k) : 0.f;
    }
}

// one 16x4 group of the soft-OR product (shared by the forward and the backward's first pass)
template <bool MASK_O>
__device__ __forceinline__ void prod_group(float2& acc_p, float2 g, bool pco, float2 mo) {
    if (MASK_O) {
        if (pco) acc_p = __ffma2_rn(__fmul2_rn(neg2(g), mo), acc_p, acc_p);          // p -= p * g * m
    } else {
        acc_p = __ffma2_rn(neg2(g), acc_p, acc_p);                                    // p *= (1 - g)
    }
}

// sum and/or soft-OR product of one 16x16 tile over the staged candidates that touch it (bit k of tm: candidate k)
template <bool SUM, bool SOFTOR, bool MASK_O, typename Stage>
__device__ __forceinline__ void accumulate_tile(const Stage& st, unsigned tm, int n, float cf, int h, const WtConsts& fc,
                                                float2 (&acc_s)[4], float2 (&acc_p)[4]) {
    constexpr bool SCALED = StageTraits<Stage>::acc;                                  // backward stages hold d^2 * s2
    while (tm) {                                                                      // warp-uniform
        const int k = __ffs(tm) - 1;
        tm &= tm - 1;
        const float2 cd = *reinterpret_cast<const float2*>(&st.cand[k]);
        const float dx = cf - cd.x;
        const float dx2 = SCALED ? __fmul_rn(dx, dx) * fc.s2 : __fmul_rn(dx, dx);
        const float ec = fabsf(cf - cd.y);
        const bool pcs = ec <= fc.hs, pco = ec <= fc.ho;
        const float4* tA = &st.tabA[k][h];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float4 A = tA[2 * i];
            const float2 d2 = __fadd2_rn(bc(dx2), make_float2(A.x, A.y));            // dc*dc + dr*dr, as the reference
            const float2 t = SCALED ? __fmul2_rn(neg2(d2), d2) : __fmul2_rn(__fmul2_rn(d2, d2), bc(fc.K2));
            const float2 g = make_float2(ex2_approx(t.x), ex2_approx(t.y));
            if (SUM) { if (pcs) acc_s[i] = __ffma2_rn(g, make_float2(A.z, A.w), acc_s[i]); }
            if (SOFTOR) {
                float2 mo = bc(1.f);
                if (MASK_O) { const float4 Bq = st.tabB4[k][2 * i + h]; mo = make_float2(Bq.z, Bq.w); }
                prod_group<MASK_O>(acc_p[i], g, pco, mo);
            }
        }
    }
}

// writes one finished 16x16 tile
template <bool SUM, bool SOFTOR, bool SUM_T>
__device__ __forceinline__ void store_tile(const RasterParams& q, const WtCoord& w, const TilePtr& tp, int j,
                                           const float2 (&acc_s)[4], const float2 (&acc_p)[4]) {
    const int ct = w.c0 + WT * j, c = ct + w.lc;
    const bool interior = w.r0 + WT <= q.ts1 && ct + WT <= q.ts0;
    float v[8];
    if (SOFTOR) {
#pragma unroll
        for (int i = 0; i < 4; ++i) { v[2 * i] = 1.f - acc_p[i].x; v[2 * i + 1] = 1.f - acc_p[i].y; }
        store_natural(q.out_softor + tp.nat + WT * j, q, w, c, interior, v);
    }
    if (SUM) {
#pragma unroll
        for (int i = 0; i < 4; ++i) { v[2 * i] = acc_s[i].x; v[2 * i + 1] = acc_s[i].y; }
        if (SUM_T) {
            float run[8];
            rows_to_run(v, run, w.h);
            store_run(q.out_sum + tp.tr + (size_t)(WT * j) * q.ts1, q, w, c, interior, run);
        } else {
            store_natural(q.out_sum + tp.nat + WT * j, q, w, c, interior, v);
        }
    }
}

// sign(d) * m for a positive m given by its bits: d's sign bit moved onto m, zero for d == 0 (and for NaN).  Written with bit
// operations and one select: the `d > 0 ? m : (d < 0 ? -m : 0)` form compiled into a divergent branch per texel (16 per tile,
// 16 % of the fused L1 backward's instructions and most of its branch-resolving stalls; profiles/r01m).
__device__ __forceinline__ float sign_times(float d, unsigned m_bits) {
    const float v = __uint_as_float((__float_as_uint(d) & 0x80000000u) | m_bits);
    return fabsf(d) > 0.f ? v : 0.f;
}

// The strip of super tiles a warp owns, and its list offsets (one load for the whole strip).
struct Strip {
    int b, bin, c0, sty0, nst, lane, tv, bx;
};
template <int WARPS, int S = WT_S>
__device__ __forceinline__ bool strip_init(Strip& s, const RasterParams& q) {
    s.b = blockIdx.z;
    const int bx = blockIdx.x, by = blockIdx.y;
    s.bin = q.shared_pattern ? 0 : s.b;
    s.lane = threadIdx.x & 31;
    // one-warp CTAs: the warp index is the constant 0, which keeps the row coordinate of the TMA boxes in uniform registers
    // (derived from threadIdx it costs a R2UR waterfall loop per box)
    s.sty0 = (by * WARPS + (WARPS == 1 ? 0 : (int)(threadIdx.x >> 5))) * S;
    if (s.sty0 >= q.tgy) return false;
    s.nst = min(S, q.tgy - s.sty0);
    s.c0 = bx * (4 * WT);
    s.bx = bx;
    const int* toff = q.tile_off + (size_t)s.bin * (q.T + 1) + (size_t)s.sty0 * q.tgx + bx;
    s.tv = 0;
    if (s.lane < 2 * s.nst) s.tv = __ldg(toff + (s.lane >> 1) * q.tgx + (s.lane & 1));   // lane 2k: begin, lane 2k+1: end of super tile k
    return true;
}

template <bool SUM, bool SOFTOR, bool SUM_T, bool MASK_O>
__global__ void __launch_bounds__(WT_CTA, FWD_MINB) splat_fwd_wt(RasterParams q, WtConsts fc) {
    typedef WarpStage<MASK_O ? 2 : 0> Stage;
    __shared__ Stage stage[WT_WARPS];
    Strip sp;
    if (!strip_init<WT_WARPS>(sp, q)) return;              // whole warp; no block-level barriers below
    Stage& st = stage[threadIdx.x >> 5];
    const Entry* entries = q.entries + (size_t)sp.bin * q.cap;
    WtCoord w;
    w.b = sp.b; w.c0 = sp.c0; w.lc = sp.lane & 15; w.h = sp.lane >> 4;
    int n = __shfl_sync(0xffffffffu, sp.tv, 1) - __shfl_sync(0xffffffffu, sp.tv, 0);
    prefetch_entries(st.raw[0], entries + __shfl_sync(0xffffffffu, sp.tv, 0), n <= WCH ? n : 0, sp.lane);

    for (int s = 0; s < sp.nst; ++s) {
        const EntryRegs e = take_entry(st.raw[s & 1], n <= WCH ? n : 0, sp.lane);
        // candidate records of the next super tile: in flight while this one is computed
        int nn = 0;
        if (s + 1 < sp.nst) {
            const int nb = __shfl_sync(0xffffffffu, sp.tv, 2 * s + 2);
            nn = __shfl_sync(0xffffffffu, sp.tv, 2 * s + 3) - nb;
            prefetch_entries(st.raw[(s + 1) & 1], entries + nb, nn <= WCH ? nn : 0, sp.lane);
        }
        if (n <= WCH) {                                    // larger lists belong to the overflow kernel
            w.r0 = (sp.sty0 + s) * WT;
            const WtMasks mk = stage_regs(st, e, n, w.c0, (float)w.r0, fc, sp.lane);
            const TilePtr tp = tile_ptr(q, w);
            for (int j = 0; j < 4; ++j) {
                const int ct = w.c0 + WT * j;
                if (ct >= q.ts0) break;
                float2 acc_s[4], acc_p[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) { acc_s[i] = bc(0.f); acc_p[i] = bc(1.f); }
                accumulate_tile<SUM, SOFTOR, MASK_O>(st, tile_mask(mk, j), n, (float)(ct + w.lc), w.h, fc, acc_s, acc_p);
                store_tile<SUM, SOFTOR, SUM_T>(q, w, tp, j, acc_s, acc_p);      // every texel of the tile is written exactly once
            }
        }
        n = nn;
    }
}

// TMA-store forward.  Same arithmetic as splat_fwd_wt; a finished 16x16 tile is parked in the warp's shared-memory
// buffers (soft-OR in natural order, the sum either natural or, for the [ts0, ts1] layout, as [column][row] with the
// 64-byte swizzle so that a lane's row-pair writes are conflict free) and leaves as one cp.async.bulk.tensor store
// per output: no per-lane addresses, no edge path (the TMA unit clips boxes at the texture border).  In splat_fwd_wt
// the stores and their address arithmetic were 130 of the ~340 instructions per tile.
template <bool SUM, bool SOFTOR, bool SUM_T, bool MASK_O>
__global__ void __launch_bounds__(WF_CTA, WF_MINB) splat_fwd_tma(RasterParams q, WtConsts fc, const __grid_constant__ CUtensorMap tm_s,
                                                                      const __grid_constant__ CUtensorMap tm_o) {
    typedef WarpStage<MASK_O ? 2 : 0> Stage;
    extern __shared__ __align__(1024) unsigned char wt_smem_ftma[];
    Strip sp;
    if (!strip_init<WF_WARPS, WF_S>(sp, q)) return;        // whole warp; no block-level barriers below
    const int wid = threadIdx.x >> 5;
    unsigned char* tout = wt_smem_ftma + wid * (2 * TMA_TILE_BYTES);         // [softor | sum], 1 KB each, 1 KB aligned
    Stage& st = reinterpret_cast<Stage*>(wt_smem_ftma + WF_WARPS * 2 * TMA_TILE_BYTES)[wid];
    const Entry* entries = q.entries + (size_t)sp.bin * q.cap;
    WtCoord w;
    w.b = sp.b; w.c0 = sp.c0; w.lc = sp.lane & 15; w.h = sp.lane >> 4;
    float* nat = reinterpret_cast<float*>(tout) + (2 * w.h) * WT + w.lc;
    const unsigned tr_base = (unsigned)(TMA_TILE_BYTES + w.lc * 64 + 8 * w.h), tr_x = (unsigned)((w.lc >> 1) & 3) << 4;
    int n = __shfl_sync(0xffffffffu, sp.tv, 1) - __shfl_sync(0xffffffffu, sp.tv, 0);
    prefetch_entries(st.raw[0], entries + __shfl_sync(0xffffffffu, sp.tv, 0), n <= WCH ? n : 0, sp.lane);

    for (int s = 0; s < sp.nst; ++s) {
        const EntryRegs e = take_entry(st.raw[s & 1], n <= WCH ? n : 0, sp.lane);
        int nn = 0;
        if (s + 1 < sp.nst) {
            const int nb = __shfl_sync(0xffffffffu, sp.tv, 2 * s + 2);
            nn = __shfl_sync(0xffffffffu, sp.tv, 2 * s + 3) - nb;
            prefetch_entries(st.raw[(s + 1) & 1], entries + nb, nn <= WCH ? nn : 0, sp.lane);
        }
        if (n <= WCH) {                                    // larger lists belong to the overflow kernel
            w.r0 = (sp.sty0 + s) * WT;
            const WtMasks mk = stage_regs(st, e, n, w.c0, (float)w.r0, fc, sp.lane);
#pragma unroll 1
            for (int j = 0; j < 4; ++j) {
                const int ct = w.c0 + WT * j;
                if (ct >= q.ts0) break;
                float2 acc_s[4], acc_p[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) { acc_s[i] = bc(0.f); acc_p[i] = bc(1.f); }
                accumulate_tile<SUM, SOFTOR, MASK_O>(st, tile_mask(mk, j), n, (float)(ct + w.lc), w.h, fc, acc_s, acc_p);
                if (tma::elect_one()) tma::store_wait_read<0>();   // the previous tile's boxes have left the buffers
                __syncwarp();
                if (SOFTOR) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) { nat[(4 * i) * WT] = 1.f - acc_p[i].x; nat[(4 * i + 1) * WT] = 1.f - acc_p[i].y; }
                }
                if (SUM) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        if (SUM_T) *reinterpret_cast<float2*>(tout + (tr_base + (tr_x ^ (unsigned)(i << 4)))) = acc_s[i];
                        else { nat[WT * WT + (4 * i) * WT] = acc_s[i].x; nat[WT * WT + (4 * i + 1) * WT] = acc_s[i].y; }
                    }
                }
                tma::fence_async_smem();
                __syncwarp();
                if (tma::elect_one()) {
                    if (SOFTOR) tma::store_3d(&tm_o, tout, ct, w.r0, w.b);
                    if (SUM) {
                        if (SUM_T) tma::store_3d(&tm_s, tout + TMA_TILE_BYTES, w.r0, ct, w.b);
                        else tma::store_3d(&tm_s, tout + TMA_TILE_BYTES, ct, w.r0, w.b);
                    }
                    tma::store_commit();
                }
            }
        }
        n = nn;
    }
    if (tma::elect_one()) tma::store_wait_read<0>();   // shared memory must outlive the last boxes
}

// Backward.  dL/dg = gS * m_s + gO * m_o * prod / (1 - g) per (texel, point); dg/dP = 4 g d2 (c - P) / sigma^2.
// SAVED: the forward's soft-OR output is available, prod = 1 - O; otherwise a first pass rebuilds prod.
// 1 - g is evaluated as (1 + 2^-23) - g so that a point sitting on a texel centre (g = 1) gives a finite
// quotient; the texel's weight g*d2*(c - P) vanishes there, and the bias is <= 1.2e-7 relative elsewhere.
// Each (candidate, tile) partial is folded once across the half warps (lanes 0-15 then hold d/dp0 parts, lanes 16-31
// d/dp1 parts) and parked in shared memory; flush_warp sums a candidate's 16 parts in one lane, all candidates at once.
// FARV: every g of the tile is below 2^-8: gO * prod * g / (1 - g) = gp * (g + g^2 + g^3) to 6e-8 relative, no reciprocal.
template <bool SUM, bool SOFTOR, bool MASK_O, bool FARV, typename Stage>
__device__ __forceinline__ void weigh_tile(Stage& st, unsigned tm, int n, float cf, int h, int lane, const WtConsts& fc,
                                           const float2 (&gs)[4], const float2 (&gp)[4]) {
    while (tm) {
        const int k = __ffs(tm) - 1;
        tm &= tm - 1;
        const float2 cd = *reinterpret_cast<const float2*>(&st.cand[k]);
        const float dx = cf - cd.x;
        const float dx2 = __fmul_rn(dx, dx) * fc.s2;
        const float ec = fabsf(cf - cd.y);
        const bool pcs = ec <= fc.hs, pco = ec <= fc.ho;
        const float4* tA = &st.tabA[k][h];
        float2 a0 = bc(0.f), a1 = bc(0.f);
        if (!MASK_O) {
            // staged over the four row groups: all exponentials, then all reciprocals, then the FMA tail -- the special-function
            // latencies overlap instead of being waited for group by group (the ncu source view showed ~400 stall samples on
            // every first consumer of a MUFU result in the group-serial schedule)
            float2 d2[4], g[4], x[4];
            float4 A[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                A[i] = tA[2 * i];
                d2[i] = __fadd2_rn(bc(dx2), make_float2(A[i].x, A[i].y));
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 t = __fmul2_rn(neg2(d2[i]), d2[i]);
                g[i] = make_float2(ex2_approx_v(t.x), ex2_approx_v(t.y));
            }
            if (FARV) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    x[i] = bc(0.f);
                    if (SOFTOR) x[i] = __fmul2_rn(gp[i], __ffma2_rn(g[i], __ffma2_rn(g[i], g[i], g[i]), g[i]));
                    if (SUM) { if (pcs) x[i] = __ffma2_rn(__fmul2_rn(gs[i], make_float2(A[i].z, A[i].w)), g[i], x[i]); }
                }
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    x[i] = bc(0.f);
                    if (SOFTOR) {
                        const float2 om = __fadd2_rn(bc(fc.c1), neg2(g[i]));
                        x[i] = make_float2(rcp_approx_v(om.x), rcp_approx_v(om.y));
                    }
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if (SOFTOR) x[i] = __fmul2_rn(gp[i], x[i]);                       // gO * prod_{m != n}(1 - g_m)
                    if (SUM) { if (pcs) x[i] = __ffma2_rn(gs[i], make_float2(A[i].z, A[i].w), x[i]); }
                    x[i] = __fmul2_rn(x[i], g[i]);
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 dy = st.tabB2[k][2 * i + h];
                const float2 wgt = __fmul2_rn(x[i], d2[i]);
                a0 = __ffma2_rn(wgt, bc(dx), a0);
                a1 = __ffma2_rn(wgt, dy, a1);
            }
        } else
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float4 A = tA[2 * i];
            float4 Bq;
            if (MASK_O) Bq = st.tabB4[k][2 * i + h];
            else { const float2 dy = st.tabB2[k][2 * i + h]; Bq = make_float4(dy.x, dy.y, 1.f, 1.f); }
            const float2 d2 = __fadd2_rn(bc(dx2), make_float2(A.x, A.y));            // d^2 * s2
            const float2 t = __fmul2_rn(neg2(d2), d2);
            const float2 g = make_float2(ex2_approx(t.x), ex2_approx(t.y));
            if (FARV && !MASK_O) {
                float2 x = bc(0.f);
                if (SOFTOR) x = __fmul2_rn(gp[i], __ffma2_rn(g, __ffma2_rn(g, g, g), g));
                if (SUM) { if (pcs) x = __ffma2_rn(__fmul2_rn(gs[i], make_float2(A.z, A.w)), g, x); }
                const float2 wgt = __fmul2_rn(x, d2);
                a0 = __ffma2_rn(wgt, bc(dx), a0);
                a1 = __ffma2_rn(wgt, make_float2(Bq.x, Bq.y), a1);
                continue;
            }
            float2 coef = bc(0.f);
            if (SOFTOR) {
                if (MASK_O) {
                    const float2 mm = pco ? make_float2(Bq.z, Bq.w) : bc(0.f);
                    const float2 om = __ffma2_rn(neg2(g), mm, bc(fc.c1));
                    coef = __fmul2_rn(__fmul2_rn(gp[i], mm), make_float2(rcp_approx(om.x), rcp_approx(om.y)));
                } else {
                    const float2 om = __fadd2_rn(bc(fc.c1), neg2(g));
                    coef = __fmul2_rn(gp[i], make_float2(rcp_approx(om.x), rcp_approx(om.y)));   // gO * prod_{m != n}(1 - g_m)
                }
            }
            if (SUM) { if (pcs) coef = __ffma2_rn(gs[i], make_float2(A.z, A.w), coef); }
            const float2 wgt = __fmul2_rn(__fmul2_rn(coef, g), d2);
            a0 = __ffma2_rn(wgt, bc(dx), a0);
            a1 = __ffma2_rn(wgt, make_float2(Bq.x, Bq.y), a1);
        }
        const float s0 = a0.x + a0.y, s1 = a1.x + a1.y;
        const float keep = h ? s1 : s0, give = h ? s0 : s1;
        st.acc[k][lane] += keep + __shfl_xor_sync(0xffffffffu, give, 16);
    }
}

// lane k (k < n) sums candidate k's d/dp0 parts, lane 16 + k its d/dp1 parts; one atomic each
template <typename Stage>
__device__ __forceinline__ void flush_warp(const Stage& st, int n, int h, int lc, float kh, float* __restrict__ dp) {
    __syncwarp();
    if (lc < n) {
        const float* a = &st.acc[lc][16 * h];
        float x = 0.f, y = 0.f;
#pragma unroll
        for (int j = 0; j < 16; j += 2) { x += a[j]; y += a[j + 1]; }
        const float val = (x + y) * kh;
        if (val != 0.f) atomicAdd(dp + (size_t)__float_as_int(st.cand[lc].z) * 2, val);
    }
}

// raw upstream values of one tile, as loaded (the transposed sum gradient still in run order)
struct TileIn {
    float s[8], o[8], sv[8];       // members a kernel variant does not use are never touched and cost no registers
};
template <bool SUM, bool SOFTOR, bool SUM_T, bool SAVED>
__device__ __forceinline__ void load_tile_in(TileIn& t, const RasterParams& q, const WtCoord& w, const TilePtr& tp, int j) {
    const int ct = w.c0 + WT * j, c = ct + w.lc;
    const bool interior = w.r0 + WT <= q.ts1 && ct + WT <= q.ts0;
    if (SUM) {
        if (SUM_T) load_run(q.g_sum + tp.tr + (size_t)(WT * j) * q.ts1, q, w, c, interior, t.s);
        else load_natural(q.g_sum + tp.nat + WT * j, q, w, c, interior, t.s);
    }
    if (SOFTOR) {
        load_natural(q.g_softor + tp.nat + WT * j, q, w, c, interior, t.o);
        if (SAVED) load_natural(q.saved_softor + tp.nat + WT * j, q, w, c, interior, t.sv);
    }
}
// upstream gradients of this lane's 8 texels: gs = gS, gp = gO (* prod when the forward's output is at hand)
template <bool SUM, bool SOFTOR, bool SUM_T, bool SAVED>
__device__ __forceinline__ void unpack_tile_in(const TileIn& in, int h, float2 (&gs)[4], float2 (&gp)[4]) {
    if (SUM) {
        float v[8];
        if (SUM_T) run_to_rows(in.s, v, h);
#pragma unroll
        for (int i = 0; i < 4; ++i) gs[i] = SUM_T ? make_float2(v[2 * i], v[2 * i + 1]) : make_float2(in.s[2 * i], in.s[2 * i + 1]);
    }
    if (SOFTOR) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            gp[i] = make_float2(in.o[2 * i], in.o[2 * i + 1]);
            if (SAVED) gp[i] = __fmul2_rn(gp[i], make_float2(1.f - in.sv[2 * i], 1.f - in.sv[2 * i + 1]));
        }
    }
}

// asynchronous copy of one natural-layout 16x16 tile into a padded shared buffer (interior tiles with 16-byte aligned
// rows), or a guarded synchronous fill with the same layout otherwise
__device__ __forceinline__ void stage_tile_async(float (&buf)[WT][24], const float* __restrict__ src, const RasterParams& q,
                                                 const WtCoord& w, int ct, int lane) {
    const bool interior = w.r0 + WT <= q.ts1 && ct + WT <= q.ts0;
    const float* org = src + ((size_t)w.b * q.ts1 + w.r0) * q.ts0 + ct;
    if (interior && (q.ts0 & 3) == 0 && (reinterpret_cast<size_t>(src) & 15) == 0) {
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            const int row = (lane >> 2) + 8 * t, ch = (lane & 3) * 4;
            const unsigned dst = (unsigned)__cvta_generic_to_shared(&buf[row][ch]);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(org + (size_t)row * q.ts0 + ch) : "memory");
        }
    } else {
        const int c = ct + w.lc, rb = 2 * w.h;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int r = rb + 4 * i + j;
                buf[r][w.lc] = (c < q.ts0 && w.r0 + r < q.ts1) ? __ldg(org + (size_t)r * q.ts0 + w.lc) : 0.f;
            }
    }
}

template <bool SUM, bool SOFTOR, bool SUM_T, bool MASK_O, bool SAVED>
__global__ void __launch_bounds__(WB_CTA, BWD_MINB) splat_bwd_wt(RasterParams q, WtConsts fc) {
    typedef WarpStage<MASK_O ? 2 : 1, true, true, 1> Stage;
    extern __shared__ __align__(16) unsigned char wt_smem[];
    Strip sp;
    if (!strip_init<WB_WARPS>(sp, q)) return;
    Stage& st = reinterpret_cast<Stage*>(wt_smem)[threadIdx.x >> 5];
    const Entry* entries = q.entries + (size_t)sp.bin * q.cap;
    WtCoord w;
    w.b = sp.b; w.c0 = sp.c0; w.lc = sp.lane & 15; w.h = sp.lane >> 4;
    const float inv_s2 = q.rcp_sigma * q.rcp_sigma;
    const float kh = 4.f * (w.h ? (float)q.ts1 : (float)q.ts0) * inv_s2 * fc.rs2;     // lanes 0-15 report d/dp0, lanes 16-31 d/dp1; rs2 undoes the table scaling
    float* dp = q.d_pts + (size_t)sp.b * q.N * 2 + w.h;
    int n = __shfl_sync(0xffffffffu, sp.tv, 1) - __shfl_sync(0xffffffffu, sp.tv, 0);
    prefetch_entries(st.raw[0], entries + __shfl_sync(0xffffffffu, sp.tv, 0), n <= WCH ? n : 0, sp.lane);
    float sraw[8];                                          // upstream sum gradient of the tile in flight (registers)
    bool have = false;                                      // tile 0 of the current super tile is already in flight

    // puts one tile's upstream values in flight: soft-OR gradient (+ saved output) through cp.async, sum gradient in registers
    auto issue = [&](const WtCoord& wc, int j) {
        const int ct = wc.c0 + WT * j;
        if (SOFTOR) {
            stage_tile_async(st.tin[0], q.g_softor, q, wc, ct, sp.lane);
            if (SAVED) stage_tile_async(st.tin[1], q.saved_softor, q, wc, ct, sp.lane);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        if (SUM) {
            const TilePtr tp = tile_ptr(q, wc);
            const bool interior = wc.r0 + WT <= q.ts1 && ct + WT <= q.ts0;
            if (SUM_T) load_run(q.g_sum + tp.tr + (size_t)(WT * j) * q.ts1, q, wc, ct + wc.lc, interior, sraw);
            else load_natural(q.g_sum + tp.nat + WT * j, q, wc, ct + wc.lc, interior, sraw);
        }
    };

    for (int s = 0; s < sp.nst; ++s) {
        const EntryRegs e = take_entry(st.raw[0], n <= WCH ? n : 0, sp.lane);
        __syncwarp();                                       // every lane holds its record: the buffer may be refilled
        int nn = 0;
        if (s + 1 < sp.nst) {
            const int nb = __shfl_sync(0xffffffffu, sp.tv, 2 * s + 2);
            nn = __shfl_sync(0xffffffffu, sp.tv, 2 * s + 3) - nb;
            prefetch_entries(st.raw[0], entries + nb, nn <= WCH ? nn : 0, sp.lane);
        }
        const bool next_live = nn > 0 && nn <= WCH;
        if (n > 0 && n <= WCH) {                           // empty: nothing to do; larger lists: overflow kernel
            w.r0 = (sp.sty0 + s) * WT;
            if (!have) issue(w, 0);
            const WtMasks mk = stage_regs(st, e, n, w.c0, (float)w.r0, fc, sp.lane);
            for (int j = 0; j < 4; ++j) {
                const int ct = w.c0 + WT * j;
                if (ct >= q.ts0) break;
                // upstream gradients of this lane's 8 texels: gs = gS, gp = gO (* prod when the forward's output is at hand)
                float2 gs[4], gp[4];
                if (SUM) {
                    float v[8];
                    if (SUM_T) run_to_rows(sraw, v, w.h);
#pragma unroll
                    for (int i = 0; i < 4; ++i) gs[i] = SUM_T ? make_float2(v[2 * i], v[2 * i + 1]) : make_float2(sraw[2 * i], sraw[2 * i + 1]);
                }
                if (SOFTOR) {
                    asm volatile("cp.async.wait_group 0;" ::: "memory");
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int r = 4 * i + 2 * w.h;
                        gp[i] = make_float2(st.tin[0][r][w.lc], st.tin[0][r + 1][w.lc]);
                        if (SAVED) gp[i] = __fmul2_rn(gp[i], make_float2(1.f - st.tin[1][r][w.lc], 1.f - st.tin[1][r + 1][w.lc]));
                    }
                    __syncwarp();                           // buffers consumed: the next tile may land
                }
                // next tile (of this super tile, or tile 0 of the next one) in flight while this one is computed
                if (j < 3 && ct + WT < q.ts0) {
                    issue(w, j + 1);
                } else if (next_live) {
                    WtCoord wn = w;
                    wn.r0 = w.r0 + WT;
                    issue(wn, 0);
                }
                const unsigned tm = tile_mask(mk, j);
                const float cf = (float)(ct + w.lc);
                if (SOFTOR && !SAVED) {                    // pass 1 (only without the saved output): per-texel product of (1 - g)
                    float2 prod[4], unused[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) prod[i] = bc(1.f);
                    accumulate_tile<false, true, MASK_O>(st, tm, n, cf, w.h, fc, unused, prod);
#pragma unroll
                    for (int i = 0; i < 4; ++i) gp[i] = __fmul2_rn(gp[i], prod[i]);
                }
                const unsigned nm = near_mask(mk, j);
                weigh_tile<SUM, SOFTOR, MASK_O, false>(st, MASK_O ? tm : nm, n, cf, w.h, sp.lane, fc, gs, gp);
                if (!MASK_O) weigh_tile<SUM, SOFTOR, MASK_O, true>(st, tm & ~nm, n, cf, w.h, sp.lane, fc, gs, gp);
            }
            flush_warp(st, n, w.h, w.lc, kh, dp);
            have = next_live;
        } else {
            have = false;
        }
        n = nn;
    }
}

// TMA-fed backward for soft-OR windows tighter than their no-op radius (every other case takes the super-tile kernel,
// ffb_splat_st.cuh).  The ncu source view of splat_bwd_wt showed ~200 instructions of per-tile overhead around ~290 of
// splat arithmetic: at an 80-register budget the compiler re-derives block / lane coordinates and the 64-bit addresses
// of three arrays for every 16x16 tile.  Here the address generation belongs to the TMA unit: lane 0 issues one
// cp.async.bulk.tensor box {16, 16, 1} per upstream array and tile (coordinates (column, row, sample); texels beyond
// the texture arrive as zeros, so there is no edge path), completion is an mbarrier transaction count, and every lane
// reads its 8 texels per array from fixed shared-memory offsets.  The transposed sum gradient ([ts0, ts1]) uses the
// 64-byte swizzle so that a lane's (column, row pair) reads are conflict free; no shuffles are needed any more.
// One 3 KB buffer set per warp: a tile's values move to registers first, then the next tile's boxes are requested and
// land while this tile is computed.
template <bool SUM, bool SOFTOR, bool SUM_T, bool SAVED>
__global__ void __launch_bounds__(WB_CTA, BWD_MINB) splat_bwd_tma(RasterParams q, WtConsts fc, const __grid_constant__ CUtensorMap tm_gs,
                                                                  const __grid_constant__ CUtensorMap tm_go,
                                                                  const __grid_constant__ CUtensorMap tm_sv) {
    typedef WarpStage<2, true, false, 1> Stage;
    constexpr int NBUF = 3;
    extern __shared__ __align__(1024) unsigned char wt_smem_tma[];
    Strip sp;
    if (!strip_init<WB_WARPS>(sp, q)) return;
    const int wid = WB_WARPS == 1 ? 0 : (int)(threadIdx.x >> 5);
    unsigned char* tin = wt_smem_tma + wid * (NBUF * TMA_TILE_BYTES);            // [go | saved | gs], 1 KB each, 1 KB aligned
    uint64_t* bar = reinterpret_cast<uint64_t*>(wt_smem_tma + WB_WARPS * NBUF * TMA_TILE_BYTES) + wid;
    Stage& st = reinterpret_cast<Stage*>(wt_smem_tma + WB_WARPS * NBUF * TMA_TILE_BYTES + 64)[wid];
    const Entry* entries = q.entries + (size_t)sp.bin * q.cap;
    WtCoord w;
    w.b = sp.b; w.c0 = sp.c0; w.lc = sp.lane & 15; w.h = sp.lane >> 4;
    const float inv_s2 = q.rcp_sigma * q.rcp_sigma;
    const float kh = 4.f * (w.h ? (float)q.ts1 : (float)q.ts0) * inv_s2 * fc.rs2;
    float* dp = q.d_pts + (size_t)sp.b * q.N * 2 + w.h;
    if (sp.lane == 0) {
        tma::mbar_init(bar, 1);
        tma::fence_mbar_init();
    }
    __syncwarp();
    unsigned phase = 0;
    bool have = false;                                      // tile 0 of the current super tile is already in flight
    constexpr unsigned kBytes = (unsigned)TMA_TILE_BYTES * ((SOFTOR ? (SAVED ? 2 : 1) : 0) + (SUM ? 1 : 0));
    // natural tiles: texel (row 4i + 2h + j, column lc) at float (4i + j) * 16 + nat_off
    const float* nat = reinterpret_cast<const float*>(tin) + (2 * w.h) * WT + w.lc;
    // transposed tile (64-byte swizzle: 16-byte chunk index ^= (column >> 1) & 3): rows 4i + 2h + {0, 1} of column lc
    const unsigned tr_base = (unsigned)(2 * TMA_TILE_BYTES + w.lc * 64 + 8 * w.h), tr_x = (unsigned)((w.lc >> 1) & 3) << 4;

    auto issue = [&](int r0, int j) {                      // called by the converged warp
        if (tma::elect_one()) {
            const int ct = w.c0 + WT * j;
            tma::mbar_expect_tx(bar, kBytes);
            if (SOFTOR) {
                tma::load_3d(tin, &tm_go, bar, ct, r0, w.b);
                if (SAVED) tma::load_3d(tin + TMA_TILE_BYTES, &tm_sv, bar, ct, r0, w.b);
            }
            if (SUM) {
                if (SUM_T) tma::load_3d(tin + 2 * TMA_TILE_BYTES, &tm_gs, bar, r0, ct, w.b);
                else tma::load_3d(tin + 2 * TMA_TILE_BYTES, &tm_gs, bar, ct, r0, w.b);
            }
        }
    };
    // dense patterns: the first tile's boxes are requested before the list bounds and the candidate records arrive -- three
    // dependent memory latencies at the head of a warp's life become one
    if (q.eager) {
        issue(sp.sty0 * WT, 0);
        have = true;
    }
    int n = __shfl_sync(0xffffffffu, sp.tv, 1) - __shfl_sync(0xffffffffu, sp.tv, 0);
    prefetch_entries(st.raw[0], entries + __shfl_sync(0xffffffffu, sp.tv, 0), n <= WCH ? n : 0, sp.lane);

    for (int s = 0; s < sp.nst; ++s) {
        const EntryRegs e = take_entry(st.raw[0], n <= WCH ? n : 0, sp.lane);
        __syncwarp();                                       // every lane holds its record: the buffer may be refilled
        int nn = 0;
        if (s + 1 < sp.nst) {
            const int nb = __shfl_sync(0xffffffffu, sp.tv, 2 * s + 2);
            nn = __shfl_sync(0xffffffffu, sp.tv, 2 * s + 3) - nb;
            prefetch_entries(st.raw[0], entries + nb, nn <= WCH ? nn : 0, sp.lane);
        }
        const bool next_live = nn > 0 && nn <= WCH;
        if (n > 0 && n <= WCH) {                           // empty: no gradient work; larger lists: overflow kernel
            w.r0 = (sp.sty0 + s) * WT;
            if (!have) issue(w.r0, 0);
            const WtMasks mk = stage_regs(st, e, n, w.c0, (float)w.r0, fc, sp.lane);
#pragma unroll 1
            for (int j = 0; j < 4; ++j) {
                float2 gs[4], gp[4];
                tma::mbar_wait(bar, phase);
                phase ^= 1u;
                if (SOFTOR) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        gp[i] = make_float2(nat[(4 * i) * WT], nat[(4 * i + 1) * WT]);
                        if (SAVED) gp[i] = __fmul2_rn(gp[i], make_float2(1.f - nat[WT * WT + (4 * i) * WT], 1.f - nat[WT * WT + (4 * i + 1) * WT]));
                    }
                }
                if (SUM) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        if (SUM_T) gs[i] = *reinterpret_cast<const float2*>(tin + (tr_base + (tr_x ^ (unsigned)(i << 4))));
                        else gs[i] = make_float2(nat[2 * WT * WT + (4 * i) * WT], nat[2 * WT * WT + (4 * i + 1) * WT]);
                    }
                }
                __syncwarp();                               // buffers consumed: the next tile may land
                // next tile (of this super tile, or tile 0 of the next one) in flight while this one is computed
                if (j < 3) issue(w.r0, j + 1);
                else if (next_live) issue(w.r0 + WT, 0);
                const unsigned tm = tile_mask(mk, j);
                const float cf = (float)(w.c0 + WT * j + w.lc);
                if (SOFTOR && !SAVED) {                    // pass 1 (only without the saved output): per-texel product of (1 - g)
                    float2 prod[4], unused[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) prod[i] = bc(1.f);
                    accumulate_tile<false, true, true>(st, tm, n, cf, w.h, fc, unused, prod);
#pragma unroll
                    for (int i = 0; i < 4; ++i) gp[i] = __fmul2_rn(gp[i], prod[i]);
                }
                weigh_tile<SUM, SOFTOR, true, false>(st, tm, n, cf, w.h, sp.lane, fc, gs, gp);
            }
            flush_warp(st, n, w.h, w.lc, kh, dp);
            have = next_live;
        } else {
            if (have) {                                     // requested eagerly, not needed: let the boxes land before the buffers go away
                tma::mbar_wait(bar, phase);
                phase ^= 1u;
            }
            have = false;
        }
        n = nn;
    }
}

// ---- overflow: super tiles whose list is longer than one chunk ---------------------------------------------------------
// The binning kernel appends such super tiles to a list; these kernels walk it with a small fixed grid, one warp per
// (super tile, sample), staging 16 candidates at a time.  Same arithmetic, no prefetching.
struct OvfParams {
    const int* count;          // number of overflow super tiles (device)
    const int* list;           // bin * T + super tile
    int B;
};
__device__ __forceinline__ bool ovf_item(const RasterParams& q, const OvfParams& o, long long it, WtCoord& w, int& bin, int& stile) {
    const int cnt = __ldg(o.count);
    const long long items = (long long)cnt * (q.shared_pattern ? o.B : 1);
    if (it >= items) return false;
    const int li = (int)(it % cnt);
    const int code = __ldg(o.list + li);
    bin = code / q.T;
    stile = code - bin * q.T;
    w.b = q.shared_pattern ? (int)(it / cnt) : bin;
    w.c0 = (stile % q.tgx) * (4 * WT);
    w.r0 = (stile / q.tgx) * WT;
    w.lc = threadIdx.x & 15;
    w.h = (threadIdx.x & 31) >> 4;
    return true;
}

template <bool SUM, bool SOFTOR, bool SUM_T, bool MASK_O>
__global__ void __launch_bounds__(WT_CTA) splat_fwd_ovf(RasterParams q, WtConsts fc, OvfParams o) {
    typedef WarpStage<MASK_O ? 2 : 0> Stage;
    __shared__ Stage stage[WT_WARPS];
    Stage& st = stage[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const long long nwarps = (long long)gridDim.x * WT_WARPS;
    for (long long it = (long long)blockIdx.x * WT_WARPS + (threadIdx.x >> 5);; it += nwarps) {
        WtCoord w;
        int bin, stile;
        if (!ovf_item(q, o, it, w, bin, stile)) break;
        const int* toff = q.tile_off + (size_t)bin * (q.T + 1) + stile;
        const int beg = __ldg(toff), end = __ldg(toff + 1);
        const Entry* entries = q.entries + (size_t)bin * q.cap;
        const TilePtr tp = tile_ptr(q, w);
        for (int j = 0; j < 4; ++j) {
            const int ct = w.c0 + WT * j;
            if (ct >= q.ts0) break;
            float2 acc_s[4], acc_p[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { acc_s[i] = bc(0.f); acc_p[i] = bc(1.f); }
            for (int base = beg; base < end; base += WCH) {
                const int n = min(WCH, end - base);
                const WtMasks mk = stage_regs(st, load_entry(entries, base, n, lane), n, w.c0, (float)w.r0, fc, lane);
                accumulate_tile<SUM, SOFTOR, MASK_O>(st, tile_mask(mk, j), n, (float)(ct + w.lc), w.h, fc, acc_s, acc_p);
            }
            store_tile<SUM, SOFTOR, SUM_T>(q, w, tp, j, acc_s, acc_p);
        }
    }
}

template <bool SUM, bool SOFTOR, bool SUM_T, bool MASK_O, bool SAVED, bool LOSS = false>
__global__ void __launch_bounds__(WT_CTA) splat_bwd_ovf(RasterParams q, WtConsts fc, OvfParams o) {
    typedef WarpStage<MASK_O ? 2 : 1, true, false, 1> Stage;
    extern __shared__ __align__(16) unsigned char wt_smem[];
    Stage& st = reinterpret_cast<Stage*>(wt_smem)[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const float inv_s2 = q.rcp_sigma * q.rcp_sigma;
    const long long nwarps = (long long)gridDim.x * WT_WARPS;
    for (long long it = (long long)blockIdx.x * WT_WARPS + (threadIdx.x >> 5);; it += nwarps) {
        WtCoord w;
        int bin, stile;
        if (!ovf_item(q, o, it, w, bin, stile)) break;
        const int* toff = q.tile_off + (size_t)bin * (q.T + 1) + stile;
        const int beg = __ldg(toff), end = __ldg(toff + 1);
        const Entry* entries = q.entries + (size_t)bin * q.cap;
        const TilePtr tp = tile_ptr(q, w);
        const float kh = 4.f * (w.h ? (float)q.ts1 : (float)q.ts0) * inv_s2 * fc.rs2;
        float* dp = q.d_pts + (size_t)w.b * q.N * 2 + w.h;
        for (int j = 0; j < 4; ++j) {
            const int ct = w.c0 + WT * j;
            if (ct >= q.ts0) break;
            const float cf = (float)(ct + w.lc);
            TileIn in;
            float2 gs[4], gp[4];
            if (LOSS) {
                // gradients of mean|softor - sum| from the forward's outputs (g_softor = softor, g_sum = sum as stored); the loss
                // value itself is accumulated by the main kernel, which visits every tile
                const int c = ct + w.lc;
                const bool interior = w.r0 + WT <= q.ts1 && ct + WT <= q.ts0;
                float sn[8], srun[8], orun[8];
                load_natural(q.g_softor + tp.nat + WT * j, q, w, c, interior, in.o);
                load_natural(q.g_sum + tp.nat + WT * j, q, w, c, interior, sn);
                const unsigned inv_bits = __float_as_uint(q.loss_inv);
                auto sgn = [&](float d) { return sign_times(d, inv_bits); };
                if (SUM_T) {
                    load_run(q.g_sum + tp.tr + (size_t)(WT * j) * q.ts1, q, w, c, interior, srun);
                    load_run(q.g_softor + tp.tr + (size_t)(WT * j) * q.ts1, q, w, c, interior, orun);
                    run_to_rows(srun, in.s, w.h);
                    run_to_rows(orun, in.sv, w.h);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float2 sg = make_float2(sgn(in.o[2 * i] - sn[2 * i]), sgn(in.o[2 * i + 1] - sn[2 * i + 1]));
                    gp[i] = __fmul2_rn(sg, make_float2(1.f - in.o[2 * i], 1.f - in.o[2 * i + 1]));
                    gs[i] = SUM_T ? make_float2(-sgn(in.sv[2 * i] - in.s[2 * i]), -sgn(in.sv[2 * i + 1] - in.s[2 * i + 1])) : neg2(sg);
                }
            } else {
                load_tile_in<SUM, SOFTOR, SUM_T, SAVED>(in, q, w, tp, j);
                unpack_tile_in<SUM, SOFTOR, SUM_T, SAVED>(in, w.h, gs, gp);
            }
            if (SOFTOR && !SAVED) {
                float2 prod[4], unused[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) prod[i] = bc(1.f);
                for (int base = beg; base < end; base += WCH) {
                    const int n = min(WCH, end - base);
                    const WtMasks mk = stage_regs(st, load_entry(entries, base, n, lane), n, w.c0, (float)w.r0, fc, lane);
                    accumulate_tile<false, true, MASK_O>(st, tile_mask(mk, j), n, cf, w.h, fc, unused, prod);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) gp[i] = __fmul2_rn(gp[i], prod[i]);
            }
            for (int base = beg; base < end; base += WCH) {
                const int n = min(WCH, end - base);
                const WtMasks mk = stage_regs(st, load_entry(entries, base, n, lane), n, w.c0, (float)w.r0, fc, lane);
                weigh_tile<SUM, SOFTOR, MASK_O, false>(st, tile_mask(mk, j), n, cf, w.h, lane, fc, gs, gp);
                flush_warp(st, n, w.h, w.lc, kh, dp);
            }
        }
    }
}
