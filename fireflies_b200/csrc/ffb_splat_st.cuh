// Super-tile backward (included by ffb_splat.cu inside namespace ffb::splat, after ffb_splat_wt.cuh).
//
// What the round-1 captures of splat_bwd_tma said (profiles/r01n): the kernel is instruction bound -- 1860 warp
// instructions per 64x16 super tile, of which ~640 are the (candidate, tile) inner loop, ~410 once-per-super-tile staging
// (a (candidate, row) table of 3 KB filled and re-read, parked partial sums zeroed and flushed) and ~700 once-per-tile work
// (four mbarrier rounds of three 16x16 boxes, 20 scalar LDS, the gO * (1 - O) products) -- and it moves 12 B/texel (both
// upstream gradients plus the saved soft-OR output) where 8 are compulsory, which alone puts its DRAM time at the
// measured copy bandwidth above 2.0 ms per 256 samples.
//
// This kernel changes the three things that follow from that:
//   * ONE request round per super tile: two {32, 16} boxes (128-byte rows, 128-byte swizzle) per natural array and one
//     {16, 64} box (64-byte swizzle) for the transposed sum gradient land on one mbarrier; the whole 64x16 block of both
//     upstream arrays is resident in shared memory (8 KB per warp) before the first texel is touched.
//   * ROW-FIXED lanes: lane = (q, cg) owns rows {q, q + 8} and columns 4 cg .. 4 cg + 3 of every 16x16 tile, so that a lane's
//     two rows are the same for the whole super tile: everything that depends on (candidate, row) is three packed
//     instructions per visit from a 16-byte record instead of a shared-memory table (3 KB less per warp, no fill pass),
//     a tile's upstream values are two conflict-free LDS.128 per natural array (8 LDS.32 for the transposed one), and the
//     packed fp32 pipe works on column pairs of one row, which is the register order those loads deliver.
//   * the soft-OR product is REBUILT (pass 1 over the tile's candidates, 5 instructions per texel pair) instead of read back
//     from the forward's output: 8 B/texel of DRAM traffic = the algorithmic bytes.  Tiles with a single candidate need
//     neither the product nor the reciprocal (the exclusive product is 1), and tiles with two candidates take each other's
//     factor directly.  The rebuilt product is also what torch.prod's backward uses (1 - O from an fp32 O loses the product's
//     bits in saturated regions).
// Kept from splat_bwd_tma: one-warp CTAs, one super tile per warp, warp-uniform tile masks from ballots, the near / far
// split (g < 2^-8: 1/(1-g) as a polynomial on the FMA pipe), g = 2^-(d2 s)^2 with pre-scaled distances, one atomic per
// (candidate, super tile, component), the overflow kernel for lists longer than WCH.  The per-candidate partial sums are no
// longer parked in shared memory (2.1 KB per warp, a zeroing pass and a 16-load flush): a visit's two sums are reduced over the
// warp with five shuffles, software-pipelined into the next visit, and accumulated in the register of the lane that owns the
// candidate -- 8.4 KB of shared memory per warp, 24 resident warps instead of 19.
#pragma once

constexpr int ST_MINB = 22;               // register target of the allocation (80 registers: up to 24 one-warp CTAs per SM fit, 8.5 KB of shared memory + 1 KB reserved each); measured 0.526 / 0.542 / 0.823 ms per 64 samples at 22 / 20 / 24
constexpr int ST_BOX = 4 * WT * WT * 4;   // one 64x16 fp32 block = 4 KB

enum StMode { ST_REBUILD, ST_LOSS };

template <bool SUM, bool SOFTOR, bool SUM_T, int MODE>
struct StSmem {
    static constexpr int n_box = MODE == ST_LOSS ? 2 : ((SOFTOR ? 1 : 0) + (SUM ? 1 : 0));
    static constexpr int off_go = 0;                                   // LOSS: the soft-OR output at the tile's own index
    static constexpr int off_gs = MODE == ST_LOSS ? ST_BOX : (SOFTOR ? ST_BOX : 0);       // LOSS: the sum output at the tile's own index (as stored)
    // LOSS + SUM_T: the same two boxes first hold the outputs at the MIRRORED index (soft-OR in off_go, sum in off_gs, {16,32} boxes),
    // from which the lane keeps one sign per texel, and then the outputs at the tile's own index
    static constexpr int off_bar = n_box * ST_BOX;
    static constexpr int off_rec = off_bar + 16;
    static constexpr int off_idx = off_rec + WCH * 16;
    // LOSS + SUM_T: -sign(softor - sum) at the mirrored index, [column 64][row 16] as int8 with a 16-byte pitch (1 KB per warp: 22 resident
    // warps per SM, where the sign as bf16 with a 40-byte pitch took 2.5 KB and allowed 19)
    static constexpr int off_sgn = off_idx + WCH * 4;
    static constexpr int sgn_pitch = 16;
    static constexpr int bytes = off_sgn + ((MODE == ST_LOSS && SUM_T) ? 4 * WT * sgn_pitch : 0);
};

// Everything is measured in units of 1 / r1 (r1 = sqrt(s2)) relative to the super tile's first texel, so that d2s = dxs^2 + dys^2 feeds
// ex2 directly (g = 2^-(d2s^2)) and a visit's distances are one packed subtraction per row pair / column pair: the record holds
// (P0 - c0) r1 and (P1 - r0) r1 (differences of nearby numbers, exact before the scaling), the lane holds its rows and columns times r1.
struct StLane {
    float2 rabs;           // the lane's two rows (q, q + 8) times r1
    float cbs;             // the lane's first column (4 cg) times r1
    unsigned nat_e;        // byte offset of (row q, columns 4 cg ..) in a natural half box for even tiles (odd tiles: ^ 64; row q + 8: + 1024; tiles 2, 3: + 2048)
    unsigned tA0;          // transposed box: byte offset of (column 4 cg, row q); column + 1: + 64; columns + 2, + 3: (^ 16) + 128 / + 192; row q + 8: ^ 32; tile j: + 1024 j
};
__device__ __forceinline__ StLane st_lane(int lane, const WtConsts& fc) {
    StLane ln;
    const int qy = lane & 7, cg = lane >> 3;
    const float sc = fc.r1;
    ln.rabs = make_float2((float)qy * sc, (float)(qy + 8) * sc);
    ln.cbs = (float)(4 * cg) * sc;
    ln.nat_e = (unsigned)(qy * 128 + ((cg ^ qy) << 4));
    ln.tA0 = (unsigned)(4 * cg) * 64u + (((unsigned)(qy >> 2) ^ ((unsigned)(cg & 1) << 1)) << 4) + (unsigned)(qy & 3) * 4u;
    // opaque to the optimiser: otherwise these are re-derived from the lane index for every tile (~25 instructions per tile)
    asm volatile("" : "+r"(ln.nat_e), "+r"(ln.tA0), "+f"(ln.cbs), "+f"(ln.rabs.x), "+f"(ln.rabs.y));
    return ln;
}
struct StTileCols {
    float2 c01, c23;       // the lane's four columns of this tile times r1
};

// geometry of one candidate {P0s, P1s, D0s, D1s} against the lane's two rows / four columns.  MSK: the sum window cuts texels that matter
// (D = (P - window origin) r1, so that dxs + D0s is the integer column offset from the window origin times r1)
struct StRow {
    float2 dys, dy2;
    bool pa, pb;           // rows inside the sum window
};
template <bool MSK>
__device__ __forceinline__ StRow st_row(const float4 rc, const StLane& ln, const WtConsts& fc) {
    StRow r;
    r.dys = __fadd2_rn(ln.rabs, bc(-rc.y));
    r.dy2 = __fmul2_rn(r.dys, r.dys);
    r.pa = r.pb = true;
    if (MSK) {
        const float2 er = __fadd2_rn(r.dys, bc(rc.w));
        r.pa = fabsf(er.x) <= fc.hs_r;
        r.pb = fabsf(er.y) <= fc.hs_r;
    }
    return r;
}
struct StCol {
    float2 dxs[2], mc[2];
};
template <bool MSK>
__device__ __forceinline__ StCol st_col(const float4 rc, const StTileCols& tc, const WtConsts& fc) {
    StCol c;
    c.dxs[0] = __fadd2_rn(tc.c01, bc(-rc.x));
    c.dxs[1] = __fadd2_rn(tc.c23, bc(-rc.x));
    if (MSK) {
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            const float2 e = __fadd2_rn(c.dxs[p], bc(rc.z));
            c.mc[p] = make_float2(__saturatef(fmaf(fabsf(e.x), fc.m_r, fc.thr_r)), __saturatef(fmaf(fabsf(e.y), fc.m_r, fc.thr_r)));
        }
    }
    return c;
}
// d2s of texel pair v (0 = row a columns 0,1; 1 = row a columns 2,3; 2, 3 = row b)
__device__ __forceinline__ float2 st_d2(const StRow& r, const StCol& c, int v) {
    return __ffma2_rn(c.dxs[v & 1], c.dxs[v & 1], bc(v < 2 ? r.dy2.x : r.dy2.y));
}

// shared-memory reads by 32-bit shared-space address: through generic pointers every access re-derives the shared window base
// (S2R SR_CgaCtaId + shifts, ~4 instructions each, ~60 per item)
__device__ __forceinline__ float4 st_lds128(unsigned a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ float2 st_lds64(unsigned a) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ float st_lds32(unsigned a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}

// highest candidate of a tile mask (bfind = one FLO; the ffs form is BREV + FLO, both on the special-function pipe)
__device__ __forceinline__ int st_next(unsigned& tm) {
    int k;
    asm("bfind.u32 %0, %1;" : "=r"(k) : "r"(tm));
    tm ^= 1u << k;
    return k;
}
// Candidate walk with the next record in flight: the chain  mask -> bfind -> address -> LDS -> first subtraction  (~80 cycles) used to sit
// at the head of every iteration, where nothing else of the iteration can start (a third of the stall samples of the pass-1 loop).
#define FFB_ST_WALK_BEGIN(tm_, rec_)                                  \
    {                                                                 \
        unsigned w_tm = (tm_);                                        \
        int k = st_next(w_tm);                                        \
        float4 rc = st_lds128((rec_) + 16u * (unsigned)k);            \
        for (;;) {                                                    \
            const bool w_more = w_tm != 0u;                           \
            int w_kn = k;                                             \
            float4 w_rcn = rc;                                        \
            if (w_more) {                                             \
                w_kn = st_next(w_tm);                                 \
                w_rcn = st_lds128((rec_) + 16u * (unsigned)w_kn);     \
            }
#define FFB_ST_WALK_END                                               \
            if (!w_more) break;                                       \
            k = w_kn;                                                 \
            rc = w_rcn;                                               \
        }                                                             \
    }

// pass 1: p *= (1 - g) over the candidates of the tile
__device__ __forceinline__ void st_prod(unsigned rec, unsigned tm, const StTileCols& tc, const StLane& ln, const WtConsts& fc, float2 (&p)[4]) {
    if (tm == 0u) return;
    FFB_ST_WALK_BEGIN(tm, rec)
        const StRow r = st_row<false>(rc, ln, fc);
        const StCol c = st_col<false>(rc, tc, fc);
        float2 g[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const float2 d2 = st_d2(r, c, v);
            const float2 t = __fmul2_rn(neg2(d2), d2);
            g[v] = make_float2(ex2_approx(t.x), ex2_approx(t.y));
        }
#pragma unroll
        for (int v = 0; v < 4; ++v) p[v] = __ffma2_rn(neg2(g[v]), p[v], p[v]);
    FFB_ST_WALK_END
}

// g of one candidate on the lane's 8 texels (two-candidate tiles keep both)
__device__ __forceinline__ void st_g(const float4 rc, const StTileCols& tc, const StLane& ln, const WtConsts& fc, float2 (&g)[4]) {
    const StRow r = st_row<false>(rc, ln, fc);
    const StCol c = st_col<false>(rc, tc, fc);
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        const float2 d2 = st_d2(r, c, v);
        const float2 t = __fmul2_rn(neg2(d2), d2);
        g[v] = make_float2(ex2_approx(t.x), ex2_approx(t.y));
    }
}

// d/dP partial sums of the previous visit, reduced over the warp while the next visit computes: the five dependent shuffles sit at the
// top of the next loop body, where the scheduler interleaves them with that visit's independent geometry and exponentials.  After the
// fold across the half warps lanes 0-15 hold d/dp0 parts and lanes 16-31 d/dp1 parts; lane (k, h) owns candidate k's component h.
struct StPend {
    float s0, s1;
    int k;
};
__device__ __forceinline__ void st_reduce(const StPend& pd, float& accr, int lane) {
    const bool up = lane >= 16;
    const float keep = up ? pd.s1 : pd.s0, give = up ? pd.s0 : pd.s1;
    float v = keep + __shfl_xor_sync(0xffffffffu, give, 16);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    if ((lane & 15) == pd.k) accr += v;
}
__device__ __forceinline__ void st_park(StPend& pd, int k, const float2 a0, const float2 a1) {
    pd.s0 = a0.x + a0.y;
    pd.s1 = a1.x + a1.y;
    pd.k = k;
}

// KIND 0: near (exclusive product = P / (1 - g) with a reciprocal), 1: far (every g < 2^-8: polynomial), 2: gp already is the
// exclusive product times gO (single-candidate tiles: gp = gO).  Without MSK the sum gradient is one addend of the same FFMA2.
template <bool SUM, bool SOFTOR, bool MSK, int KIND>
__device__ __forceinline__ void st_weigh(unsigned rec, StPend& pd, float& accr, unsigned tm, const StTileCols& tc, const StLane& ln,
                                         int lane, const WtConsts& fc, const float2 (&gs)[4], const float2 (&gp)[4]) {
    if (tm == 0u) return;
    FFB_ST_WALK_BEGIN(tm, rec)
        st_reduce(pd, accr, lane);
        const StRow r = st_row<SUM && MSK>(rc, ln, fc);
        const StCol c = st_col<SUM && MSK>(rc, tc, fc);
        float2 d2[4], g[4], x[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            d2[v] = st_d2(r, c, v);
            const float2 t = __fmul2_rn(neg2(d2[v]), d2[v]);
            g[v] = make_float2(ex2_approx_v(t.x), ex2_approx_v(t.y));
        }
        if (KIND == 0 && SOFTOR) {
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                const float2 om = __fadd2_rn(bc(fc.c1), neg2(g[v]));
                x[v] = make_float2(rcp_approx_v(om.x), rcp_approx_v(om.y));
            }
        }
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const bool pr = v < 2 ? r.pa : r.pb;
            float2 e = bc(1.f);                                                       // 1 / (1 - g)
            if (SOFTOR && KIND == 0) e = x[v];
            if (SOFTOR && KIND == 1) e = __ffma2_rn(g[v], __ffma2_rn(g[v], g[v], bc(1.f)), bc(1.f));   // 1 + g + g^2 (+ O(g^3) < 6e-8)
            if (!SOFTOR) x[v] = bc(0.f);
            else if (KIND == 2) x[v] = gp[v];
            else if (SUM && !MSK) x[v] = __ffma2_rn(gp[v], e, gs[v]);                 // gO * prod_{m != n}(1 - g_m) + gS
            else x[v] = __fmul2_rn(gp[v], e);
            if (SUM && MSK) { if (pr) x[v] = __ffma2_rn(gs[v], c.mc[v & 1], x[v]); }
            if (SUM && !MSK && (!SOFTOR || KIND == 2)) x[v] = __fadd2_rn(x[v], gs[v]);   // loop invariant: hoisted
            x[v] = __fmul2_rn(x[v], g[v]);
        }
        float2 a0 = bc(0.f), a1 = bc(0.f);
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const float2 wgt = __fmul2_rn(x[v], d2[v]);
            a0 = __ffma2_rn(wgt, c.dxs[v & 1], a0);
            a1 = __ffma2_rn(wgt, bc(v < 2 ? r.dys.x : r.dys.y), a1);
        }
        st_park(pd, k, a0, a1);
    FFB_ST_WALK_END
}

// two-candidate tile: the exclusive product of one candidate is the other's factor
template <bool SUM, bool MSK>
__device__ __forceinline__ void st_weigh_one_of_pair(const float4 rc, StPend& pd, float& accr, int k, const StTileCols& tc, const StLane& ln,
                                                     int lane, const WtConsts& fc, const float2 (&gs)[4], const float2 (&go)[4],
                                                     const float2 (&gn)[4], const float2 (&gm)[4]) {
    st_reduce(pd, accr, lane);
    const StRow r = st_row<SUM && MSK>(rc, ln, fc);
    const StCol c = st_col<SUM && MSK>(rc, tc, fc);
    float2 a0 = bc(0.f), a1 = bc(0.f);
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        const float2 d2 = st_d2(r, c, v);
        float2 x = __ffma2_rn(neg2(gm[v]), go[v], (SUM && !MSK) ? __fadd2_rn(go[v], gs[v]) : go[v]);   // gO * (1 - g_other) [+ gS]
        const bool pr = v < 2 ? r.pa : r.pb;
        if (SUM && MSK) { if (pr) x = __ffma2_rn(gs[v], c.mc[v & 1], x); }
        const float2 wgt = __fmul2_rn(__fmul2_rn(x, gn[v]), d2);
        a0 = __ffma2_rn(wgt, c.dxs[v & 1], a0);
        a1 = __ffma2_rn(wgt, bc(v < 2 ? r.dys.x : r.dys.y), a1);
    }
    st_park(pd, k, a0, a1);
}
template <bool SUM, bool MSK>
__device__ __forceinline__ void st_weigh_pair(unsigned rec, StPend& pd, float& accr, unsigned tm, const StTileCols& tc, const StLane& ln,
                                              int lane, const WtConsts& fc, const float2 (&gs)[4], const float2 (&go)[4]) {
    const int k0 = __ffs(tm) - 1, k1 = 31 - __clz(tm);
    const float4 rc0 = st_lds128(rec + 16u * (unsigned)k0), rc1 = st_lds128(rec + 16u * (unsigned)k1);
    float2 g0[4], g1[4];
    st_g(rc0, tc, ln, fc, g0);
    st_g(rc1, tc, ln, fc, g1);
    st_weigh_one_of_pair<SUM, MSK>(rc0, pd, accr, k0, tc, ln, lane, fc, gs, go, g0, g1);
    st_weigh_one_of_pair<SUM, MSK>(rc1, pd, accr, k1, tc, ln, lane, fc, gs, go, g1, g0);
}

// three-candidate tile (the most frequent kind: 22 % of the tiles at config 3): the three sets of exponentials stay in registers, a
// candidate's exclusive product is the other two factors -- no pass 1, no reciprocal, 24 instead of ~50 special-function ops
template <bool SUM, bool MSK>
__device__ __forceinline__ void st_weigh_one_of_triple(const float4 rc, StPend& pd, float& accr, int k, const StTileCols& tc, const StLane& ln,
                                                       int lane, const WtConsts& fc, const float2 (&gs)[4], const float2 (&go)[4],
                                                       const float2 (&gn)[4], const float2 (&ga)[4], const float2 (&gb)[4]) {
    st_reduce(pd, accr, lane);
    const StRow r = st_row<SUM && MSK>(rc, ln, fc);
    const StCol c = st_col<SUM && MSK>(rc, tc, fc);
    float2 a0 = bc(0.f), a1 = bc(0.f);
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        const float2 d2 = st_d2(r, c, v);
        const float2 e1 = __ffma2_rn(neg2(ga[v]), go[v], go[v]);                      // gO * (1 - g_a)
        float2 x = __ffma2_rn(neg2(gb[v]), e1, (SUM && !MSK) ? __fadd2_rn(e1, gs[v]) : e1);   // gO * (1 - g_a)(1 - g_b) [+ gS]
        const bool pr = v < 2 ? r.pa : r.pb;
        if (SUM && MSK) { if (pr) x = __ffma2_rn(gs[v], c.mc[v & 1], x); }
        const float2 wgt = __fmul2_rn(__fmul2_rn(x, gn[v]), d2);
        a0 = __ffma2_rn(wgt, c.dxs[v & 1], a0);
        a1 = __ffma2_rn(wgt, bc(v < 2 ? r.dys.x : r.dys.y), a1);
    }
    st_park(pd, k, a0, a1);
}
template <bool SUM, bool MSK>
__device__ __forceinline__ void st_weigh_triple(unsigned rec, StPend& pd, float& accr, unsigned tm, const StTileCols& tc, const StLane& ln,
                                                int lane, const WtConsts& fc, const float2 (&gs)[4], const float2 (&go)[4]) {
    const int k0 = st_next(tm), k1 = st_next(tm), k2 = st_next(tm);
    const float4 rc0 = st_lds128(rec + 16u * (unsigned)k0), rc1 = st_lds128(rec + 16u * (unsigned)k1), rc2 = st_lds128(rec + 16u * (unsigned)k2);
    float2 g0[4], g1[4], g2[4];
    st_g(rc0, tc, ln, fc, g0);
    st_g(rc1, tc, ln, fc, g1);
    st_g(rc2, tc, ln, fc, g2);
    st_weigh_one_of_triple<SUM, MSK>(rc0, pd, accr, k0, tc, ln, lane, fc, gs, go, g0, g1, g2);
    st_weigh_one_of_triple<SUM, MSK>(rc1, pd, accr, k1, tc, ln, lane, fc, gs, go, g1, g0, g2);
    st_weigh_one_of_triple<SUM, MSK>(rc2, pd, accr, k2, tc, ln, lane, fc, gs, go, g2, g0, g1);
}

// tile with NK candidates (four: st_tile): each exponential once per texel, each candidate's exclusive product from a prefix product
// (forward over the candidates) times a suffix product (backward) -- no pass 1, no reciprocal, and the product stays the one
// torch.prod's backward forms.  NK candidates' g of all 8 texels do not fit in registers, so the work is blocked over the lane's four
// texel pairs: per pair, NK values of g and of the prefix; the candidates' partial sums are carried across the pairs and then reduced
// one visit per candidate, in the walk order of st_weigh.  The geometry is recomputed in the backward sweep rather than kept.
// The upstream values are read pair by pair (up(v, gs, go)): all four pairs held through the sweeps would spill.
template <bool SUM, bool MSK, int NK, class Up>
__device__ __forceinline__ void st_weigh_few(unsigned rec, StPend& pd, float& accr, unsigned tm, const StTileCols& tc, const StLane& ln,
                                             int lane, const WtConsts& fc, const Up& up) {
    int kn[NK];
    float4 rc[NK];
#pragma unroll
    for (int n = 0; n < NK; ++n) {
        kn[n] = st_next(tm);
        rc[n] = st_lds128(rec + 16u * (unsigned)kn[n]);
    }
    float a0[NK], a1[NK];                                                             // the lane's d/dp0, d/dp1 parts of candidate n
#pragma unroll
    for (int n = 0; n < NK; ++n) a0[n] = a1[n] = 0.f;
#pragma unroll 1
    for (int v = 0; v < 4; ++v) {
        const float2 cx = (v & 1) ? tc.c23 : tc.c01;
        const float ry = v < 2 ? ln.rabs.x : ln.rabs.y;
        float2 gs = bc(0.f), p;
        up(v, gs, p);                                                                 // p: gO * prod_{m < n}(1 - g_m)
        float2 g[NK], pre[NK];
#pragma unroll
        for (int n = 0; n < NK; ++n) {
            const float2 dxs = __fadd2_rn(cx, bc(-rc[n].x));
            const float dys = ry - rc[n].y;
            const float2 d2 = __ffma2_rn(dxs, dxs, bc(dys * dys));
            const float2 t = __fmul2_rn(neg2(d2), d2);
            g[n] = make_float2(ex2_approx(t.x), ex2_approx(t.y));
            pre[n] = p;
            if (n + 1 < NK) p = __ffma2_rn(neg2(g[n]), p, p);
        }
        float2 suf = bc(1.f);                                                         // prod_{m > n}(1 - g_m)
#pragma unroll
        for (int n = NK - 1; n >= 0; --n) {
            const float2 dxs = __fadd2_rn(cx, bc(-rc[n].x));
            const float dys = ry - rc[n].y;
            const float2 d2 = __ffma2_rn(dxs, dxs, bc(dys * dys));
            float2 x;                                                                 // gO * prod_{m != n}(1 - g_m) [+ gS]
            if (SUM && !MSK) x = __ffma2_rn(pre[n], suf, gs);
            else x = __fmul2_rn(pre[n], suf);
            if (SUM && MSK) {
                if (fabsf(dys + rc[n].w) <= fc.hs_r) {
                    const float2 e = __fadd2_rn(dxs, bc(rc[n].z));
                    const float2 mc = make_float2(__saturatef(fmaf(fabsf(e.x), fc.m_r, fc.thr_r)), __saturatef(fmaf(fabsf(e.y), fc.m_r, fc.thr_r)));
                    x = __ffma2_rn(gs, mc, x);
                }
            }
            if (n > 0) suf = __ffma2_rn(neg2(g[n]), suf, suf);
            const float2 wgt = __fmul2_rn(__fmul2_rn(x, g[n]), d2);
            const float s0 = fmaf(wgt.y, dxs.y, wgt.x * dxs.x), s1 = (wgt.x + wgt.y) * dys;
            a0[n] += s0;
            a1[n] += s1;
        }
    }
#pragma unroll
    for (int n = 0; n < NK; ++n) {
        st_reduce(pd, accr, lane);
        pd.s0 = a0[n]; pd.s1 = a1[n]; pd.k = kn[n];
    }
}

// ---- staging: one candidate per lane -> tile masks (ballots) and 16-byte records {(P0 - c0) r1, (P1 - r0) r1, (P0 - f0) r1, (P1 - f1) r1} ----
__device__ __forceinline__ WtMasks st_stage(const RasterParams& q, const WtConsts& fc, int bin, int beg, int n, int c0, int r0, int lane,
                                            float4* rec, int* idx) {
    const float r0f = (float)r0, c0f = (float)c0;
    bool ta[4] = {false, false, false, false}, na[4] = {false, false, false, false};
    if (lane < n) {
        const float4 ea = __ldg(reinterpret_cast<const float4*>(q.entries + (size_t)bin * q.cap + beg + lane));
        const uint4 eb = __ldg(reinterpret_cast<const uint4*>(q.entries + (size_t)bin * q.cap + beg + lane) + 1);
        const int clo = (int)(eb.y & 0xffff) - c0, chi = (int)(eb.y >> 16) - c0;
        const float px = ea.x - c0f, py = ea.y - r0f;       // relative to the super tile (exact: differences of nearby numbers)
        const float ry = fmaxf(fmaxf(-py, py - (float)(WT - 1)), 0.f);
        const float ry2 = ry * ry;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            // a tile whose nearest texel centre has g < 1e-7 contributes nothing measurable to d/dP (weights g * d2 * (c - P); wt_consts)
            const float xl = (float)(WT * i);
            const float rx = fmaxf(fmaxf(xl - px, px - (xl + (float)(WT - 1))), 0.f);
            const float rr = fmaf(rx, rx, ry2);
            ta[i] = clo < WT * i + WT && chi > WT * i && rr <= fc.disc2;
            na[i] = ta[i] && rr < fc.near2;
        }
        rec[lane] = make_float4(px * fc.r1, py * fc.r1, (ea.x - ea.z) * fc.r1, (ea.y - ea.w) * fc.r1);
        idx[lane] = (int)eb.z;
    }
    WtMasks mk;
    mk.tb01 = __ballot_sync(0xffffffffu, ta[0]) | (__ballot_sync(0xffffffffu, ta[1]) << 16);
    mk.tb23 = __ballot_sync(0xffffffffu, ta[2]) | (__ballot_sync(0xffffffffu, ta[3]) << 16);
    mk.nb01 = __ballot_sync(0xffffffffu, na[0]) | (__ballot_sync(0xffffffffu, na[1]) << 16);
    mk.nb23 = __ballot_sync(0xffffffffu, na[2]) | (__ballot_sync(0xffffffffu, na[3]) << 16);
    return mk;
}

// LOSS + SUM_T, first request round: the boxes hold the forward's outputs at the mirrored index ({16,32} boxes: [column 64][row 16]).
// -sign(softor - sum) of all 1024 texels goes to shared memory as int8 (-1, 0, +1): lane L takes columns L and L + 32 -- four
// conflict-free LDS.128 per array and column (the 64-byte swizzle spreads the eight lanes of a phase over all banks), packed
// subtractions, and one 4-byte store per four rows.  The consumer mapping (rows q, q + 8; columns 4 cg ..) reads them back with
// conflict-free 8-bit loads.  (A first version kept two bits per texel in registers: 64 scalar loads and ~350 instructions per item.)
__device__ __forceinline__ unsigned st_sign_bf16x2(const float2 d) {
    // (sign(d.y) as bf16) << 16 | (sign(d.x) as bf16): the high halves of the two floats are d truncated to bf16 (zero only for a zero or
    // flushed difference), and sign(x) = min(max(x * 2^127, -1), 1) in packed bf16 -- four instructions per texel pair where the
    // select form took fourteen
    unsigned h, w;
    asm("prmt.b32 %0, %1, %2, 0x7632;" : "=r"(h) : "r"(__float_as_uint(d.x)), "r"(__float_as_uint(d.y)));
    asm("{\n\t.reg .b32 t;\n\tmul.rn.bf16x2 t, %1, %2;\n\tmax.bf16x2 t, t, %3;\n\tmin.bf16x2 %0, t, %4;\n\t}"
        : "=r"(w) : "r"(h), "r"(0x7f007f00u), "r"(0xbf80bf80u), "r"(0x3f803f80u));
    return w;
}
template <typename L>
__device__ __forceinline__ void st_loss_signs(unsigned sbase, int lane) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int c = lane + 32 * half;
        const unsigned row = sbase + (unsigned)c * 64u, sw = (unsigned)((c >> 1) & 3);
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
            const unsigned a = row + (((unsigned)ch ^ sw) << 4);
            const float4 o = st_lds128(a + L::off_go), m = st_lds128(a + L::off_gs);
            const unsigned w0 = st_sign_bf16x2(__fadd2_rn(make_float2(o.x, o.y), neg2(make_float2(m.x, m.y))));
            const unsigned w1 = st_sign_bf16x2(__fadd2_rn(make_float2(o.z, o.w), neg2(make_float2(m.z, m.w))));
            // four bf16 signs -> four int8 of the NEGATED sign (what the consumer needs): top bytes 0x3f / 0xbf / 0x00 (0x80 for -0)
            unsigned T;
            asm("prmt.b32 %0, %1, %2, 0x7531;" : "=r"(T) : "r"(w0), "r"(w1));
            const unsigned nz = T & 0x01010101u, sg = (T >> 7) & nz;
            const unsigned out = (nz * 0xffu) ^ (sg * 0xfeu);                          // +1 -> 0xff, -1 -> 0x01, 0 -> 0x00
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(sbase + L::off_sgn + (unsigned)c * L::sgn_pitch + (unsigned)ch * 4u), "r"(out) : "memory");
        }
    }
}
__device__ __forceinline__ float st_lds_s8(unsigned a) {
    int v;
    asm volatile("ld.shared.s8 %0, [%1];" : "=r"(v) : "r"(a));
    return (float)v;
}

// one 16x16 tile of the resident super tile: upstream values of the lane's 8 texels from shared memory, then the tile's candidates
template <bool SUM, bool SOFTOR, bool SUM_T, bool MSK, int MODE, bool FEW>
__device__ __forceinline__ void st_tile(unsigned sbase, int j, unsigned tm, unsigned nm, unsigned rec, StPend& pd, float& accr,
                                        float& lacc, const StLane& ln, int lane, const WtConsts& fc) {
    typedef StSmem<SUM, SOFTOR, SUM_T, MODE> L;
    constexpr bool LOSS = MODE == ST_LOSS;
    const unsigned nb = (ln.nat_e ^ ((unsigned)(j & 1) << 6)) + (unsigned)(j >> 1) * (ST_BOX / 2);
    float2 gs[4], gp[4];
    auto ld_nat = [&](int off, float2 (&v)[4]) {
        const float4 a = st_lds128(sbase + off + nb);
        const float4 c = st_lds128(sbase + off + nb + 1024);
        v[0] = make_float2(a.x, a.y); v[1] = make_float2(a.z, a.w); v[2] = make_float2(c.x, c.y); v[3] = make_float2(c.z, c.w);
    };
    auto ld_tr = [&](int off, float2 (&v)[4]) {
        const unsigned t = sbase + off + j * 1024;
        const unsigned a0 = t + ln.tA0, a2 = t + (ln.tA0 ^ 16u) + 128u, b0 = t + (ln.tA0 ^ 32u), b2 = t + (ln.tA0 ^ 48u) + 128u;
        v[0] = make_float2(st_lds32(a0), st_lds32(a0 + 64));
        v[1] = make_float2(st_lds32(a2), st_lds32(a2 + 64));
        v[2] = make_float2(st_lds32(b0), st_lds32(b0 + 64));
        v[3] = make_float2(st_lds32(b2), st_lds32(b2 + 64));
    };
    StTileCols tc;
    {
        const float sc = fc.r1;
        const float cfs = fmaf((float)j, (float)WT * sc, ln.cbs);
        tc.c01 = make_float2(cfs, cfs + sc);
        tc.c23 = make_float2(cfs + 2.f * sc, cfs + 3.f * sc);
    }
    const bool one = (tm & (tm - 1u)) == 0u;               // at most one candidate on this tile (warp-uniform)
    const int cands = __popc(tm);
    // four candidates (14 % of the tiles, 21 % of the visits at config 3): one pass (st_weigh_few).  Five or six spill at the
    // 80-register target, and so does the one-shot kernel with this branch (FEW = false there)
    if (FEW && !LOSS && SOFTOR && cands == 4) {
        auto up = [&](int v, float2& s, float2& o) {        // texel pair v of both upstream arrays
            const unsigned n = sbase + nb + (unsigned)(v >> 1) * 1024u + (unsigned)(v & 1) * 8u;
            o = st_lds64(n + L::off_go);
            if (SUM && SUM_T) {
                const unsigned t = sbase + L::off_gs + j * 1024;
                const unsigned a = t + ((v < 2 ? ln.tA0 : (ln.tA0 ^ 32u)) ^ ((v & 1) ? 16u : 0u));
                s = make_float2(st_lds32(a + ((v & 1) ? 128u : 0u)), st_lds32(a + ((v & 1) ? 192u : 64u)));
            } else if (SUM) {
                s = st_lds64(n + L::off_gs);
            }
        };
        st_weigh_few<SUM, MSK, 4>(rec, pd, accr, tm, tc, ln, lane, fc, up);
        return;
    }
    if (LOSS) {
        // unit signs here; the 1 / numel of the mean is folded into the final scale of d/dP and of the loss
        float2 o[4], s[4];
        ld_nat(L::off_go, o);
        ld_nat(L::off_gs, s);
        float2 lacc2 = bc(0.f);
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const float2 d = __fadd2_rn(o[v], neg2(s[v]));
            gp[v] = make_float2(sign_times(d.x, 0x3f800000u), sign_times(d.y, 0x3f800000u));      // d loss / d softor (unit)
            lacc2 = __ffma2_rn(d, gp[v], lacc2);                                                    // |d| = d * sign(d), exact
            gs[v] = neg2(gp[v]);
        }
        lacc += lacc2.x + lacc2.y;
        if (tm == 0u) return;
        if (SUM_T) {
            // d loss / d sum at this texel = -sign(softor - sum) at the mirrored texel (st_loss_signs)
            const unsigned t = sbase + L::off_sgn + (unsigned)(WT * j + 4 * (lane >> 3)) * L::sgn_pitch + (unsigned)(lane & 7);
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                const unsigned a = t + (unsigned)(2 * (v & 1)) * L::sgn_pitch + (v >> 1) * 8u;
                gs[v] = make_float2(st_lds_s8(a), st_lds_s8(a + L::sgn_pitch));
            }
        }
    } else {
        if (SUM) { if (SUM_T) ld_tr(L::off_gs, gs); else ld_nat(L::off_gs, gs); }
        if (SOFTOR) ld_nat(L::off_go, gp);
    }
    if (one || !SOFTOR) {
        st_weigh<SUM, SOFTOR, MSK, 2>(rec, pd, accr, tm, tc, ln, lane, fc, gs, gp);
        return;
    }
    if (cands == 2) {                                       // exclusive products are the other candidate's factor (no pass 1, no reciprocal)
        st_weigh_pair<SUM, MSK>(rec, pd, accr, tm, tc, ln, lane, fc, gs, gp);
        return;
    }
    if (cands == 3) {
        st_weigh_triple<SUM, MSK>(rec, pd, accr, tm, tc, ln, lane, fc, gs, gp);
        return;
    }
    if (LOSS) {
        // longer lists: gO * prod from the forward's output (resident anyway), every candidate divides its own factor out
        const unsigned nb_ = (ln.nat_e ^ ((unsigned)(j & 1) << 6)) + (unsigned)(j >> 1) * (ST_BOX / 2);
        float2 o[4];
        {
            const float4 a = st_lds128(sbase + L::off_go + nb_), c = st_lds128(sbase + L::off_go + nb_ + 1024);
            o[0] = make_float2(a.x, a.y); o[1] = make_float2(a.z, a.w); o[2] = make_float2(c.x, c.y); o[3] = make_float2(c.z, c.w);
        }
#pragma unroll
        for (int v = 0; v < 4; ++v) gp[v] = __ffma2_rn(neg2(o[v]), gp[v], gp[v]);          // sign * (1 - softor), one rounding like fl(1 - o)
        st_weigh<SUM, SOFTOR, MSK, 0>(rec, pd, accr, nm, tc, ln, lane, fc, gs, gp);
        st_weigh<SUM, SOFTOR, MSK, 1>(rec, pd, accr, tm & ~nm, tc, ln, lane, fc, gs, gp);
        return;
    }
    // pass 1 over all candidates but one, whose exponentials then serve both passes: its exclusive product is the product so far
    // (no reciprocal), and its factor completes the product for the others
    const unsigned low = tm & (0u - tm), rest = tm ^ low;
    {
        float2 p[4] = {bc(1.f), bc(1.f), bc(1.f), bc(1.f)};
        st_prod(rec, rest, tc, ln, fc, p);
        int k;
        asm("bfind.u32 %0, %1;" : "=r"(k) : "r"(low));
        const float4 rc = st_lds128(rec + 16u * (unsigned)k);
        st_reduce(pd, accr, lane);
        const StRow r = st_row<SUM && MSK>(rc, ln, fc);
        const StCol c = st_col<SUM && MSK>(rc, tc, fc);
        float2 a0 = bc(0.f), a1 = bc(0.f);
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const float2 d2 = st_d2(r, c, v);
            const float2 t = __fmul2_rn(neg2(d2), d2);
            const float2 g = make_float2(ex2_approx(t.x), ex2_approx(t.y));
            const float2 ex = __fmul2_rn(gp[v], p[v]);                                // gO * prod_{m != this}(1 - g_m)
            gp[v] = __ffma2_rn(neg2(g), ex, ex);                                      // gO * prod over all
            float2 x = ex;
            const bool pr = v < 2 ? r.pa : r.pb;
            if (SUM && MSK) { if (pr) x = __ffma2_rn(gs[v], c.mc[v & 1], x); }
            if (SUM && !MSK) x = __fadd2_rn(x, gs[v]);
            const float2 wgt = __fmul2_rn(__fmul2_rn(x, g), d2);
            a0 = __ffma2_rn(wgt, c.dxs[v & 1], a0);
            a1 = __ffma2_rn(wgt, bc(v < 2 ? r.dys.x : r.dys.y), a1);
        }
        st_park(pd, k, a0, a1);
    }
    st_weigh<SUM, SOFTOR, MSK, 0>(rec, pd, accr, rest & nm, tc, ln, lane, fc, gs, gp);
    st_weigh<SUM, SOFTOR, MSK, 1>(rec, pd, accr, rest & ~nm, tc, ln, lane, fc, gs, gp);
}

// requests half h (columns 32 h .. 32 h + 31) of the super tile at (c0, r0) of sample b: 2 KB per array on bar
template <bool SUM, bool SOFTOR, bool SUM_T, int MODE>
__device__ __forceinline__ void st_issue_half(unsigned char* st_smem, uint64_t* bar, int h, int c0, int r0, int b, const CUtensorMap* tm_gs,
                                              const CUtensorMap* tm_go, const CUtensorMap* tm_sv, const CUtensorMap* tm_ot, bool mirrored = false) {
    typedef StSmem<SUM, SOFTOR, SUM_T, MODE> L;
    constexpr bool LOSS = MODE == ST_LOSS;
    if (tma::elect_one()) {
        const int ch = c0 + 2 * WT * h, o = h * (ST_BOX / 2);
        tma::mbar_expect_tx(bar, (unsigned)(L::n_box * ST_BOX / 2));
        if (LOSS && SUM_T && mirrored) {
            tma::load_3d(st_smem + L::off_go + o, tm_ot, bar, r0, ch, b);
            tma::load_3d(st_smem + L::off_gs + o, tm_sv, bar, r0, ch, b);
            return;
        }
        if (SOFTOR || LOSS) tma::load_3d(st_smem + L::off_go + o, tm_go, bar, ch, r0, b);
        if (SUM || LOSS) {
            if (SUM_T && !LOSS) tma::load_3d(st_smem + L::off_gs + o, tm_gs, bar, r0, ch, b);
            else tma::load_3d(st_smem + L::off_gs + o, tm_gs, bar, ch, r0, b);
        }
    }
}

// the item's d/dP: lane (k, h) holds candidate k's component h
__device__ __forceinline__ float st_scale(const RasterParams& q, const WtConsts& fc, int lane) {
    return 4.f * ((lane >> 4) ? (float)q.ts1 : (float)q.ts0) * q.rcp_sigma * q.rcp_sigma * fc.rs3;
}
__device__ __forceinline__ void st_flush(const RasterParams& q, float kh, const StPend& pd, float accr, int lane, int n, int b, const int* idx) {
    st_reduce(pd, accr, lane);                              // the last visit's sums
    const int lc = lane & 15, h = lane >> 4;
    if (lc < n) {
        const float val = accr * kh;
        if (val != 0.f) atomicAdd(q.d_pts + ((size_t)b * q.N + idx[lc]) * 2 + h, val);
    }
}

// MODE ST_REBUILD: tm_gs = upstream sum gradient ([ts1,ts0] boxes {32,16}, or [ts0,ts1] boxes {16,32} when SUM_T), tm_go = upstream
// soft-OR gradient; the soft-OR product is rebuilt from the candidates.
// MODE ST_LOSS: upstream gradients of mean|softor - sum| formed from the forward's outputs (rasterization.py:589-599):
// tm_go = soft-OR output, tm_gs = sum output addressed like the soft-OR output (its own index: [ts0,ts1] read as stored),
// and for SUM_T tm_sv / tm_ot = sum / soft-OR outputs as {16,32} boxes at the mirrored index (a first request round into the same
// two boxes: 8.5 KB of shared memory per warp like the other mode, where four resident boxes allowed only 13 warps per SM).
//
// One-shot form (sparse patterns, !q.eager, where most super tiles are empty; ST_REBUILD only): one one-warp CTA per (super tile,
// sample), and nothing is requested for super tiles without candidates.
template <bool SUM, bool SOFTOR, bool SUM_T, bool MSK>
__global__ void __launch_bounds__(32, ST_MINB) splat_bwd_st(RasterParams q, WtConsts fc, const __grid_constant__ CUtensorMap tm_gs,
                                                            const __grid_constant__ CUtensorMap tm_go) {
    typedef StSmem<SUM, SOFTOR, SUM_T, ST_REBUILD> L;
    extern __shared__ __align__(1024) unsigned char st_smem[];
    const int lane = threadIdx.x;
    const int bx = blockIdx.x, sty = blockIdx.y, b = blockIdx.z;
    const int bin = q.shared_pattern ? 0 : b;
    const int c0 = bx * (4 * WT), r0 = sty * WT;
    uint64_t* bar = reinterpret_cast<uint64_t*>(st_smem + L::off_bar);
    float4* rec = reinterpret_cast<float4*>(st_smem + L::off_rec);
    int* idx = reinterpret_cast<int*>(st_smem + L::off_idx);
    if (lane == 0) {
        tma::mbar_init(bar, 1);
        tma::mbar_init(bar + 1, 1);
        tma::fence_mbar_init();
    }
    __syncwarp();
    const int* toff = q.tile_off + (size_t)bin * (q.T + 1) + (size_t)sty * q.tgx + bx;
    const int beg = __ldg(toff), n = __ldg(toff + 1) - beg;
    if (n <= 0 || n > WCH) return;                          // empty: no gradient work; longer lists: overflow kernel
    st_issue_half<SUM, SOFTOR, SUM_T, ST_REBUILD>(st_smem, bar, 0, c0, r0, b, &tm_gs, &tm_go, nullptr, nullptr);
    st_issue_half<SUM, SOFTOR, SUM_T, ST_REBUILD>(st_smem, bar + 1, 1, c0, r0, b, &tm_gs, &tm_go, nullptr, nullptr);
    const StLane ln = st_lane(lane, fc);
    const unsigned sbase = tma::smem_u32(st_smem);
    const WtMasks mk = st_stage(q, fc, bin, beg, n, c0, r0, lane, rec, idx);
    StPend pd = {0.f, 0.f, 0};
    float accr = 0.f;                                       // lane (k, h): d/dp_h of candidate k, summed over the super tile
    float lacc = 0.f;
    __syncwarp();
    unsigned tbits = mk.tb01, nbits = mk.nb01;             // tile masks shifted out as the tiles go by
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
        if (j == 0) tma::mbar_wait(bar, 0);
        if (j == 2) {
            tma::mbar_wait(bar + 1, 0);
            tbits = mk.tb23; nbits = mk.nb23;
        }
        const unsigned tm = tbits & 0xffffu, nm = nbits & 0xffffu;
        tbits >>= 16; nbits >>= 16;
        if (tm == 0u) continue;
        st_tile<SUM, SOFTOR, SUM_T, MSK, ST_REBUILD, false>(sbase, j, tm, nm, sbase + L::off_rec, pd, accr, lacc, ln, lane, fc);
    }
    st_flush(q, st_scale(q, fc, lane), pd, accr, lane, n, b, idx);
}

// Pipelined item loop (dense patterns: nearly every super tile has candidates).  The one-shot kernel keeps only ~19 of its 24 warp slots
// per SM filled (a one-warp CTA lives ~7 us and its slot stays empty ~2 us until the next CTA starts), and every warp begins with two
// dependent global loads (list bounds, then records) before it can do anything.  Here a warp walks several (super tile, sample) items:
// the two halves of the upstream blocks sit behind one mbarrier each, and the next item's left half is requested as soon as tiles 0
// and 1 of the current one are done, its right half after tiles 2 and 3 -- the same 8 KB of shared memory hold a two-stage pipeline.
// The next item's list bounds are loaded a whole item ahead, its records are pulled into L1 half an item ahead.  The mode decides how
// the items are handed out (launch_bwd_stp): ST_REBUILD -- the CTA walks `chunk` consecutive items and exits, the hardware block
// scheduler balances the launch; ST_LOSS -- resident warps claim items from a global counter, two items ahead.
struct StItem {
    int b, sty, bx;
};
__device__ __forceinline__ StItem st_decode(const RasterParams& q, int it, float inv_T, float inv_tgx) {
    StItem s;
    if (q.log_T >= 0) {                                      // power-of-two tile grids (2048^2: 32 x 128 super tiles): shifts
        s.b = it >> q.log_T;
        const int rem = it & (q.T - 1);
        s.sty = rem >> q.log_tgx;
        s.bx = rem & (q.tgx - 1);
        return s;
    }
    s.b = __float2int_rz(__int2float_rn(it) * inv_T);
    int rem = it - s.b * q.T;
    if (rem < 0) { --s.b; rem += q.T; } else if (rem >= q.T) { ++s.b; rem -= q.T; }
    s.sty = __float2int_rz(__int2float_rn(rem) * inv_tgx);
    s.bx = rem - s.sty * q.tgx;
    if (s.bx < 0) { --s.sty; s.bx += q.tgx; } else if (s.bx >= q.tgx) { ++s.sty; s.bx -= q.tgx; }
    return s;
}
template <bool SUM, bool SOFTOR, bool SUM_T, bool MSK, int MODE>
__global__ void __launch_bounds__(32, ST_MINB) splat_bwd_stp(RasterParams q, WtConsts fc, const __grid_constant__ CUtensorMap tm_gs,
                                                             const __grid_constant__ CUtensorMap tm_go,
                                                             const __grid_constant__ CUtensorMap tm_sv,
                                                             const __grid_constant__ CUtensorMap tm_ot, int n_items, unsigned* counter, int chunk) {
    typedef StSmem<SUM, SOFTOR, SUM_T, MODE> L;
    constexpr bool LOSS = MODE == ST_LOSS;
    extern __shared__ __align__(1024) unsigned char st_smem[];
    const int lane = threadIdx.x;
    int it = LOSS ? (int)blockIdx.x : (int)blockIdx.x * chunk;
    if (it >= n_items) return;
    if (!LOSS) n_items = min(n_items, it + chunk);
    uint64_t* bar = reinterpret_cast<uint64_t*>(st_smem + L::off_bar);
    float4* rec = reinterpret_cast<float4*>(st_smem + L::off_rec);
    int* idx = reinterpret_cast<int*>(st_smem + L::off_idx);
    if (lane == 0) {
        tma::mbar_init(bar, 1);
        tma::mbar_init(bar + 1, 1);
        tma::fence_mbar_init();
    }
    __syncwarp();
    const float inv_T = 1.0f / (float)q.T, inv_tgx = 1.0f / (float)q.tgx;
    auto toff_of = [&](const StItem& s) { return q.tile_off + (size_t)(q.shared_pattern ? 0 : s.b) * (q.T + 1) + (size_t)s.sty * q.tgx + s.bx; };
    // LOSS claims items: the first gridDim.x items are the CTAs' own indices, the counter hands out the rest.  One lane asks (claim_ask)
    // at the start of an item; the warp picks the answer up (claim_get) at its end, a whole item of work later.
    auto claim_ask = [&]() {
        unsigned v = 0;
        if (LOSS && lane == 0) v = atomicAdd(counter, 1u);
        return v;
    };
    auto claim_get = [&](unsigned v) { return (int)__shfl_sync(0xffffffffu, v, 0) + (int)gridDim.x; };
    constexpr bool TWO = LOSS && SUM_T;                     // two request rounds per item: mirrored index (sign bits), then own index
    StItem cur = st_decode(q, it, inv_T, inv_tgx);
    st_issue_half<SUM, SOFTOR, SUM_T, MODE>(st_smem, bar, 0, cur.bx * (4 * WT), cur.sty * WT, cur.b, &tm_gs, &tm_go, &tm_sv, &tm_ot, TWO);
    st_issue_half<SUM, SOFTOR, SUM_T, MODE>(st_smem, bar + 1, 1, cur.bx * (4 * WT), cur.sty * WT, cur.b, &tm_gs, &tm_go, &tm_sv, &tm_ot, TWO);
    int nit = LOSS ? claim_get(claim_ask()) : it + 1;        // the item after this one
    int beg, end;
    {
        const int* t = toff_of(cur);
        beg = __ldg(t); end = __ldg(t + 1);
    }
    const StLane ln = st_lane(lane, fc);
    const unsigned sbase = tma::smem_u32(st_smem);
    const float kh = st_scale(q, fc, lane) * (LOSS ? q.loss_inv : 1.f);
    unsigned phase = 0;
#pragma unroll 1
    for (;;) {
        // next item: list bounds now (consumed half an item later), the item after it from the counter
        const bool more = nit < n_items;
        const StItem nx = st_decode(q, more ? nit : it, inv_T, inv_tgx);
        int nbeg = 0, nend = 0;
        if (more) {
            const int* t = toff_of(nx);
            nbeg = __ldg(t); nend = __ldg(t + 1);
        }
        const unsigned asked = more ? claim_ask() : 0u;     // the item after the next
        const int n = end - beg, c0 = cur.bx * (4 * WT), r0 = cur.sty * WT;
        const bool grad = n > 0 && n <= WCH;               // empty: no gradient work; longer lists: overflow kernel
        if (TWO) {
            // round 1 (requested during the previous item): outputs at the mirrored index -> one sign per texel; then round 2, the
            // outputs at the item's own index, lands while the candidates are staged.  Each barrier completes twice per item, so
            // the mirrored round always waits on parity 0 and the own round on parity 1.
            tma::mbar_wait(bar, 0);
            tma::mbar_wait(bar + 1, 0);
            st_loss_signs<L>(sbase, lane);
            __syncwarp();
            st_issue_half<SUM, SOFTOR, SUM_T, MODE>(st_smem, bar, 0, c0, r0, cur.b, &tm_gs, &tm_go, &tm_sv, &tm_ot);
            st_issue_half<SUM, SOFTOR, SUM_T, MODE>(st_smem, bar + 1, 1, c0, r0, cur.b, &tm_gs, &tm_go, &tm_sv, &tm_ot);
        }
        WtMasks mk;
        mk.tb01 = mk.tb23 = mk.nb01 = mk.nb23 = 0u;
        if (grad) mk = st_stage(q, fc, q.shared_pattern ? 0 : cur.b, beg, n, c0, r0, lane, rec, idx);
        StPend pd = {0.f, 0.f, 0};
        float accr = 0.f, lacc = 0.f;
        __syncwarp();
        unsigned tbits = mk.tb01, nbits = mk.nb01;
#pragma unroll 1
        for (int j = 0; j < 4; ++j) {
            if (j == 0) tma::mbar_wait(bar, TWO ? 1u : phase);
            if (j == 2) {
                __syncwarp();                               // every lane is done with the left half: the next item's may land
                if (more) {
                    st_issue_half<SUM, SOFTOR, SUM_T, MODE>(st_smem, bar, 0, nx.bx * (4 * WT), nx.sty * WT, nx.b, &tm_gs, &tm_go, &tm_sv, &tm_ot, TWO);
                    const int nn = nend - nbeg;             // the next item's records: into L1 now, loaded when its staging starts
                    if (lane < nn && nn <= WCH)
                        asm volatile("prefetch.global.L1 [%0];" ::"l"(q.entries + (size_t)(q.shared_pattern ? 0 : nx.b) * q.cap + nbeg + lane));
                }
                tma::mbar_wait(bar + 1, TWO ? 1u : phase);
                tbits = mk.tb23; nbits = mk.nb23;
            }
            const unsigned tm = tbits & 0xffffu, nm = nbits & 0xffffu;
            tbits >>= 16; nbits >>= 16;
            if (!LOSS && tm == 0u) continue;
            st_tile<SUM, SOFTOR, SUM_T, MSK, MODE, true>(sbase, j, tm, nm, sbase + L::off_rec, pd, accr, lacc, ln, lane, fc);
        }
        __syncwarp();
        if (more) st_issue_half<SUM, SOFTOR, SUM_T, MODE>(st_smem, bar + 1, 1, nx.bx * (4 * WT), nx.sty * WT, nx.b, &tm_gs, &tm_go, &tm_sv, &tm_ot, TWO);
        if (grad) st_flush(q, kh, pd, accr, lane, n, cur.b, idx);
        if (LOSS) {
            lacc = warp_sum(lacc);
            if (lane == 0) atomicAdd(q.loss + cur.b, lacc * q.loss_inv);
        }
        if (!more) break;
        it = nit; nit = LOSS ? claim_get(asked) : nit + 1; cur = nx; beg = nbeg; end = nend;
        phase ^= 1u;
        __syncwarp();                                       // records and point indices of this item are dead
    }
}
