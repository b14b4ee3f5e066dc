// Laser splat: fused splat + {sum, soft-OR} reduction, forward and backward, for sm_100a.
//
// Replaces (reference paths relative to the Fireflies tree):
//   fireflies/graphics/rasterization.py:7-37    rasterize_points     (dense [N,H,W])
//   fireflies/graphics/rasterization.py:156-161 softor / sum
//   fireflies/graphics/rasterization.py:164-472 baked_sum, baked_sum_2, baked_softor, baked_softor_2
//   + the torch autograd of those w.r.t. `points`.
//
// Design (HBM-bound gather, no tensor cores -- nothing here is a contraction):
//   * prepare: one CTA per sample bins its N points into texture tiles, lists sorted by point index so
//     accumulation order is deterministic.  Two tilings: 64x16 super tiles with 32-byte list entries for
//     the warp-tile kernels (ffb_splat_wt.cuh, the production path whenever the texture is larger than
//     the footprints), 64x32 CTA tiles with index lists for the general kernels below (textures smaller
//     than a footprint, where the reference's slice clipping is not a plain intersection).  The
//     warp-tile path bins with the one-pass kernel (slot lists and records in shared memory; the whole
//     grid at once or in bands of tile rows); count / scan / fill with one 32-byte record per point in
//     the workspace (scaled position + the integer clip windows of both reductions) is its form for
//     large N and the general path's only form.
//   * general forward: one CTA per (tile, sample).  Each warp owns 8 rows x 32 columns, a lane owns one column
//     (8 texels in registers).  Candidate records are staged in shared memory; rows outside a point's
//     window are skipped with warp-uniform branches, so only the column overhang is wasted work.  Every
//     output texel is written exactly once with 128-byte warp stores: traffic = 4 B/texel/reduction.
//   * backward: same tiling.  Pass 1 rebuilds the soft-OR product (zero factors tracked like torch.prod's
//     backward) and caches g in shared memory; pass 2 forms dL/dg per (texel, point), accumulates the two
//     partial derivatives per lane, reduces them with warp shuffles and issues one shared-memory atomic
//     per (warp, point), then one global atomic per (tile, point).
#include <stdlib.h>

#include "ffb_common.cuh"
#include "ffb_tma.cuh"

namespace ffb {
namespace splat {

constexpr int TW = 64;        // tile width  (columns, texture_size[0] axis)
constexpr int TH = 32;        // tile height (rows,    texture_size[1] axis)
constexpr int WROWS = 8;      // rows per warp
constexpr int CTA = 256;      // 8 warps: 2 column halves x 4 row groups
constexpr int CHUNK = 128;    // candidate records staged per pass
constexpr int KCACHE = 6;     // cached g slots per warp in the backward (8 rows x 32 lanes each; dynamic smem)
constexpr int PREP_CTA = 1024;
constexpr int PREP_MINB = 1;
constexpr int WT = 16;        // warp tile side of the warp-tile kernels (ffb_splat_wt.cuh)
constexpr int WCH = 16;       // candidates a warp stages at once; longer super-tile lists go to the overflow kernels.  Measured at 12 (25 resident
                              // backward warps instead of 22, but 3 % of the super tiles overflow): forward 0.403 / backward 0.625 ms against 0.382 / 0.614
static_assert(WCH <= 16 && WCH % 4 == 0, "ballot masks hold 16 bits per tile; the staging structs are 16-byte aligned per WCH rows");

struct __align__(16) PointRec {
    float p0, p1;             // points * texture_size
    uint32_t sc, sr;          // sum window:    columns lo | hi << 16, rows lo | hi << 16  (half-open)
    uint32_t oc, orow;        // soft-OR window
    uint32_t uc, ur;          // union, used for culling and binning
};
static_assert(sizeof(PointRec) == 32, "PointRec must be 32 bytes");

// list entry of the warp-tile kernels: everything a warp needs about one candidate point
struct __align__(16) Entry {
    float p0, p1;             // points * texture_size
    float f0, f1;             // window origin (integer valued): |c - f0| <= H, |r - f1| <= H
    uint32_t ur;              // union row span     lo | hi << 16  (half open)
    uint32_t uc;              // union column span  lo | hi << 16
    int32_t idx;              // point index (backward: where d/dP goes)
    uint32_t pad;
};
static_assert(sizeof(Entry) == 32, "Entry must be 32 bytes");

struct Plan {
    int Bp;                   // number of binned pattern instances (1 when the pattern is shared)
    bool fast;                // warp-tile kernels (64x16 super tiles, Entry lists) vs general kernels (64x32, index lists)
    int tw, th;               // binning tile size
    int tgx, tgy, T;          // tile grid
    int band_rows;            // tile rows binned per pass of the prepare kernel (shared-memory counters)
    int cap;                  // list capacity per instance
    size_t off_recs, off_tileoff, off_list, off_entries, off_ovf, total;
    // window parameters
    int fp_s, half_s, h_s;    // baked: fp/half ; dense: h = cut-off half width
    int fp_o, half_o, h_o;
    int H_s, H_o;             // nominal Chebyshev half widths around floor(P) (fast kernels)
    bool mask_o;              // the baked soft-OR window is tighter than its exact no-op radius
    bool fast_ok;             // texture larger than the footprints: clipping is plain intersection
};

static inline int iceil_sqrt(double x) {
    int r = (int)ceil(sqrt(x));
    return r < 1 ? 1 : r;
}

static int make_plan(const ffb_splat_desc* d, Plan* p) {
    if (!d) return fail_arg(FFB_E_ARG, "splat: null descriptor");
    if (d->B <= 0 || d->N <= 0 || d->ts0 <= 0 || d->ts1 <= 0) return fail_arg(FFB_E_ARG, "splat: B, N, ts0, ts1 must be positive");
    if (d->ts0 > 65535 || d->ts1 > 65535) return fail_arg(FFB_E_LIMIT, "splat: texture side > 65535");
    if (!(d->sigma > 0.f)) return fail_arg(FFB_E_ARG, "splat: sigma must be > 0");
    if (d->num_std_sum < 0 || d->num_std_softor < 0) return fail_arg(FFB_E_ARG, "splat: num_std must be >= 0");
    p->Bp = d->pts_batch_stride == 0 ? 1 : d->B;
    // footprint = odd(floor(sqrt(sigma)) * num_std)  (rasterization.py:180-182; sqrt in fp32 like sigma.sqrt())
    const int root = (int)floorf(sqrtf(d->sigma));
    auto fp_of = [&](int num_std, int* fp, int* half) {
        int f = root * num_std;
        if (f % 2 == 0) f += 1;
        *fp = f;
        *half = (f - 1) / 2;
    };
    fp_of(d->num_std_sum, &p->fp_s, &p->half_s);
    fp_of(d->num_std_softor, &p->fp_o, &p->half_o);
    // no-op radii: g < 1.7e-38 once (d^2/sigma)^2 > 87 ; 1-g == 1 exactly once g <= 2^-25 (u^2 >= 17.5)
    // (2% margin on d^2; exp_neg clamps at w = 87, i.e. g < 1.7e-38 is treated as 0)
    p->h_s = iceil_sqrt((double)d->sigma * sqrt(87.0) * 1.02);
    p->h_o = iceil_sqrt((double)d->sigma * sqrt(17.5) * 1.02);
    p->H_s = d->num_std_sum > 0 ? p->half_s : p->h_s;
    p->mask_o = d->num_std_softor > 0 && p->half_o < p->h_o;
    p->H_o = p->mask_o ? p->half_o : p->h_o;
    p->fast_ok = (d->num_std_sum == 0 || (d->ts0 > p->fp_s && d->ts1 > p->fp_s)) &&
                 (d->num_std_softor == 0 || (d->ts0 > p->fp_o && d->ts1 > p->fp_o));
    {
        const char* e = getenv("FFB_SPLAT_GENERAL");     // debugging / tests: force the general kernels
        p->fast = p->fast_ok && d->ts0 <= 32000 && d->ts1 <= 32000 && !(e && e[0] == '1');
    }
    p->tw = p->fast ? 4 * WT : TW;
    p->th = p->fast ? WT : TH;
    p->tgx = (d->ts0 + p->tw - 1) / p->tw;
    p->tgy = (d->ts1 + p->th - 1) / p->th;
    p->T = p->tgx * p->tgy;
    {
        const int max_tiles = 20 * 1024;                 // 2 ints of shared memory per tile of a band
        if (p->tgx > max_tiles) return fail_arg(FFB_E_LIMIT, "splat: texture too wide for the binning kernel");
        p->band_rows = max_tiles / p->tgx;
        if (p->band_rows > p->tgy) p->band_rows = p->tgy;
    }
    int w_s = d->num_std_sum > 0 ? p->fp_s : 2 * p->h_s + 1;
    int w_o = d->num_std_softor > 0 ? (p->fp_o < 2 * p->h_o + 1 ? p->fp_o : 2 * p->h_o + 1) : 2 * p->h_o + 1;
    int w = (w_s > w_o ? w_s : w_o) + 1;
    long tiles_x = (w + 1) / p->tw + 2, tiles_y = (w + 1) / p->th + 2;
    if (tiles_x > p->tgx) tiles_x = p->tgx;
    if (tiles_y > p->tgy) tiles_y = p->tgy;
    long cap = (long)d->N * tiles_x * tiles_y;
    if (cap > 0x7fffffffL) return fail_arg(FFB_E_LIMIT, "splat: tile list capacity overflows int32");
    p->cap = (int)cap;
    size_t o = 0;
    p->off_recs = o;     o += (size_t)p->Bp * d->N * sizeof(PointRec);
    o = (o + 255) & ~(size_t)255;
    p->off_tileoff = o;  o += (size_t)p->Bp * (p->T + 1) * sizeof(int);
    o = (o + 255) & ~(size_t)255;
    p->off_list = o;     o += (size_t)p->Bp * p->cap * sizeof(int);
    o = (o + 255) & ~(size_t)255;
    p->off_entries = o;  o += p->fast ? (size_t)p->Bp * p->cap * sizeof(Entry) : 0;
    o = (o + 255) & ~(size_t)255;
    p->off_ovf = o;      o += p->fast ? ((size_t)p->Bp * p->T + 1) * sizeof(int) : 0;      // [0] = count, then bin * T + super tile
    p->total = (o + 255) & ~(size_t)255;
    return 0;
}

struct PrepParams {
    const float* pts;
    long long stride;
    int N, ts0, ts1, tgx, tgy, T, cap;
    int tw, th, band_rows;   // binning tile size, tile rows per shared-memory band
    int baked_s, fp_s, half_s, h_s;
    int baked_o, fp_o, half_o, h_o;
    int h_union;      // max Chebyshev half width of the two (nominal) reduction windows
    PointRec* recs;
    int* tile_off;
    int* list;        // general kernels: point indices per tile
    Entry* entries;   // warp-tile kernels: records per super tile
    int* ovf;         // warp-tile kernels: [0] = number of super tiles with more than WCH candidates, then their codes
    int* windows;     // nullable
};

// One axis of the reference's footprint clipping (rasterization.py:186,214-230): returns [lo,hi) in texture
// indices and the (wo, rs, re) triple.
__device__ __forceinline__ void baked_axis(float P, int half, int fp, int ts, int& lo, int& hi, int& wo, int& rs, int& re) {
    const float fo = floorf(P - (float)half);
    if (!(fo > -1.0e9f && fo < 1.0e9f)) { lo = hi = 0; wo = 0; rs = 0; re = 0; return; }   // NaN / far away
    wo = (int)fo;
    rs = wo < 0 ? -wo : 0;
    wo = wo < 0 ? 0 : wo;
    re = (wo + fp >= ts) ? ts - wo : fp;
    int n = re - rs;
    n = n < 0 ? 0 : n;
    lo = wo;
    hi = wo + n;
    if (hi > ts) hi = ts;
    if (lo >= ts) { lo = hi = 0; }
}
__device__ __forceinline__ void square_axis(float P, int h, int ts, int& lo, int& hi) {
    const float fl = floorf(P);
    if (!(fl > -1.0e9f && fl < 1.0e9f)) { lo = hi = 0; return; }
    const int c = (int)fl;
    lo = c - h; hi = c + h + 1;
    lo = lo < 0 ? 0 : lo;
    hi = hi > ts ? ts : hi;
    if (hi <= lo) { lo = hi = 0; }
}
__device__ __forceinline__ uint32_t pack_win(int lo, int hi) { return (uint32_t)lo | ((uint32_t)hi << 16); }

__device__ __forceinline__ PointRec make_rec(const PrepParams& q, float x, float y, int* win /* [2][2][3] or null */) {
    PointRec r;
    r.p0 = x * (float)q.ts0;      // points.clone() * texture_size  (rasterization.py:18)
    r.p1 = y * (float)q.ts1;
    int lo[2][2], hi[2][2];       // [reduction][axis]
    const float P[2] = {r.p0, r.p1};
    const int ts[2] = {q.ts0, q.ts1};
#pragma unroll
    for (int ax = 0; ax < 2; ++ax) {
        int wo = 0, rs = 0, re = 0;
        if (q.baked_s) {
            baked_axis(P[ax], q.half_s, q.fp_s, ts[ax], lo[0][ax], hi[0][ax], wo, rs, re);
            if (win) { win[(0 * 2 + ax) * 3 + 0] = wo; win[(0 * 2 + ax) * 3 + 1] = rs; win[(0 * 2 + ax) * 3 + 2] = re; }
        } else {
            square_axis(P[ax], q.h_s, ts[ax], lo[0][ax], hi[0][ax]);
            if (win) { win[(0 * 2 + ax) * 3 + 0] = 0; win[(0 * 2 + ax) * 3 + 1] = 0; win[(0 * 2 + ax) * 3 + 2] = 0; }
        }
        int l2, h2;
        square_axis(P[ax], q.h_o, ts[ax], l2, h2);            // exact no-op bound of the soft-OR
        if (q.baked_o) {
            baked_axis(P[ax], q.half_o, q.fp_o, ts[ax], lo[1][ax], hi[1][ax], wo, rs, re);
            if (win) { win[(1 * 2 + ax) * 3 + 0] = wo; win[(1 * 2 + ax) * 3 + 1] = rs; win[(1 * 2 + ax) * 3 + 2] = re; }
            lo[1][ax] = max(lo[1][ax], l2);
            hi[1][ax] = min(hi[1][ax], h2);
            if (hi[1][ax] <= lo[1][ax]) lo[1][ax] = hi[1][ax] = 0;
        } else {
            lo[1][ax] = l2; hi[1][ax] = h2;
            if (win) { win[(1 * 2 + ax) * 3 + 0] = 0; win[(1 * 2 + ax) * 3 + 1] = 0; win[(1 * 2 + ax) * 3 + 2] = 0; }
        }
    }
    // an empty axis empties the whole window
#pragma unroll
    for (int red = 0; red < 2; ++red)
        if (hi[red][0] <= lo[red][0] || hi[red][1] <= lo[red][1]) lo[red][0] = hi[red][0] = lo[red][1] = hi[red][1] = 0;
    r.sc = pack_win(lo[0][0], hi[0][0]); r.sr = pack_win(lo[0][1], hi[0][1]);
    r.oc = pack_win(lo[1][0], hi[1][0]); r.orow = pack_win(lo[1][1], hi[1][1]);
    int ulo[2], uhi[2];
#pragma unroll
    for (int ax = 0; ax < 2; ++ax) {
        const bool es = hi[0][ax] <= lo[0][ax], eo = hi[1][ax] <= lo[1][ax];
        if (es && eo) { ulo[ax] = uhi[ax] = 0; }
        else if (es) { ulo[ax] = lo[1][ax]; uhi[ax] = hi[1][ax]; }
        else if (eo) { ulo[ax] = lo[0][ax]; uhi[ax] = hi[0][ax]; }
        else { ulo[ax] = min(lo[0][ax], lo[1][ax]); uhi[ax] = max(hi[0][ax], hi[1][ax]); }
    }
    // the fast kernels mask with the nominal squares floor(P) +- H; make sure binning/culling covers them
    // (they differ from the reference-exact windows above only when fp32 rounding of P - half crosses an integer)
#pragma unroll
    for (int ax = 0; ax < 2; ++ax) {
        int l2, h2;
        square_axis(P[ax], q.h_union, ts[ax], l2, h2);
        if (h2 > l2) {
            if (uhi[ax] <= ulo[ax]) { ulo[ax] = l2; uhi[ax] = h2; }
            else { ulo[ax] = min(ulo[ax], l2); uhi[ax] = max(uhi[ax], h2); }
        }
    }
    if (uhi[0] <= ulo[0] || uhi[1] <= ulo[1]) ulo[0] = uhi[0] = ulo[1] = uhi[1] = 0;
    r.uc = pack_win(ulo[0], uhi[0]); r.ur = pack_win(ulo[1], uhi[1]);
    return r;
}

// window origin of the warp-tile kernels' Chebyshev masks along one axis: the reference's (unclipped) slice start
// floor(P - half) plus half for a baked window (rasterization.py:186), floor(P) otherwise.  Exact for every point whose window
// can reach a texture side of up to 65535; beyond 2^22 texels (and for NaN) a far sentinel that masks every texel.  Integer valued
// and exact in fp32 (|result| < 2^23).
__device__ __forceinline__ float origin_axis_f(float P, int baked, int half) {
    const float fo = floorf(baked ? P - (float)half : P);
    if (!(fo > -4194304.f && fo < 4194304.f)) return fo > 0.f ? 4194304.f : -4194304.f;
    return baked ? fo + (float)half : fo;
}

// list entry {p0, p1, f0, f1 | ur, uc, idx, 0} as two 128-bit stores
__device__ __forceinline__ void store_entry(Entry* dst, float p0, float p1, uint32_t ur, uint32_t uc, unsigned idx, int baked, int half) {
    uint4* d = reinterpret_cast<uint4*>(dst);
    d[0] = make_uint4(__float_as_uint(p0), __float_as_uint(p1), __float_as_uint(origin_axis_f(p0, baked, half)),
                      __float_as_uint(origin_axis_f(p1, baked, half)));
    d[1] = make_uint4(ur, uc, idx, 0u);
}

// the reference's slice triples of point n ([Bp][N][2][2][3])
__device__ __forceinline__ void store_windows(const PrepParams& q, int bin, int n, const int (&win)[12]) {
    int* w = q.windows + ((size_t)bin * q.N + n) * 12;
#pragma unroll
    for (int k = 0; k < 12; ++k) w[k] = win[k];
}

// Batcher's odd-even merge sort on 16 registers (63 compare-exchanges, 0-1 principle checked exhaustively): a quarter of the
// instructions of ranking by counting; empty slots (INT_MAX) sink to the end
__device__ __forceinline__ void sort16(int (&l)[16]) {
#define FFB_CE(a, c) { const int lo_ = min(l[a], l[c]), hi_ = max(l[a], l[c]); l[a] = lo_; l[c] = hi_; }
    FFB_CE(0,1) FFB_CE(2,3) FFB_CE(0,2) FFB_CE(1,3) FFB_CE(1,2) FFB_CE(4,5) FFB_CE(6,7) FFB_CE(4,6) FFB_CE(5,7) FFB_CE(5,6)
    FFB_CE(0,4) FFB_CE(2,6) FFB_CE(2,4) FFB_CE(1,5) FFB_CE(3,7) FFB_CE(3,5) FFB_CE(1,2) FFB_CE(3,4) FFB_CE(5,6)
    FFB_CE(8,9) FFB_CE(10,11) FFB_CE(8,10) FFB_CE(9,11) FFB_CE(9,10) FFB_CE(12,13) FFB_CE(14,15) FFB_CE(12,14) FFB_CE(13,15) FFB_CE(13,14)
    FFB_CE(8,12) FFB_CE(10,14) FFB_CE(10,12) FFB_CE(9,13) FFB_CE(11,15) FFB_CE(11,13) FFB_CE(9,10) FFB_CE(11,12) FFB_CE(13,14)
    FFB_CE(0,8) FFB_CE(4,12) FFB_CE(4,8) FFB_CE(2,10) FFB_CE(6,14) FFB_CE(6,10) FFB_CE(2,4) FFB_CE(6,8) FFB_CE(10,12)
    FFB_CE(1,9) FFB_CE(5,13) FFB_CE(5,9) FFB_CE(3,11) FFB_CE(7,15) FFB_CE(7,11) FFB_CE(3,5) FFB_CE(7,9) FFB_CE(11,13)
    FFB_CE(1,2) FFB_CE(3,4) FFB_CE(5,6) FFB_CE(7,8) FFB_CE(9,10) FFB_CE(11,12) FFB_CE(13,14)
#undef FFB_CE
}

// exclusive scan of cnt[0, nt) by the whole CTA (two levels of warp shuffles): thread tid owns [beg, end) and gets base plus the
// counts before beg.  base is read after the scan's barriers.
__device__ __forceinline__ int block_exclusive_scan(const int* cnt, int nt, int* warp_tot, const int& base, int& beg, int& end) {
    const int tid = threadIdx.x;
    const int per = (nt + PREP_CTA - 1) / PREP_CTA;
    beg = min(tid * per, nt); end = min(beg + per, nt);
    int local = 0;
    for (int i = beg; i < end; ++i) local += cnt[i];
    int incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, incl, o);
        if ((tid & 31) >= o) incl += v;
    }
    if ((tid & 31) == 31) warp_tot[tid >> 5] = incl;
    __syncthreads();
    if (tid < 32) {
        int v = warp_tot[tid], sc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, sc, o);
            if (tid >= o) sc += t;
        }
        warp_tot[tid] = sc - v;
    }
    __syncthreads();
    return base + warp_tot[tid >> 5] + incl - local;
}

// One CTA per binned pattern instance: count / scan / fill with the records in the workspace.  FAST: 64x16 super tiles, 32-byte
// entries (what the warp-tile path runs when the one-pass kernel's shared arrays do not fit); otherwise 64x32 CTA tiles, index
// lists.  The tile grid is processed in bands of whole tile rows so that the counters fit in shared memory for any texture size.
template <bool FAST>
__global__ void __launch_bounds__(PREP_CTA, PREP_MINB) prepare_kernel(PrepParams q) {
    extern __shared__ __align__(16) int sm[];
    const int band_tiles = q.band_rows * q.tgx;
    int* cnt = sm;                 // [band_tiles] counts, then exclusive offsets
    int* cur = sm + band_tiles;    // [band_tiles] fill cursors
    __shared__ int warp_tot[32];
    __shared__ int band_base;
    const int bin = blockIdx.x, tid = threadIdx.x;
    const float* pts = q.pts + (long long)bin * q.stride;
    PointRec* recs = q.recs + (size_t)bin * q.N;
    int* tile_off = q.tile_off + (size_t)bin * (q.T + 1);
    int* list = q.list + (size_t)bin * q.cap;          // FAST: unsorted scratch; otherwise the final index lists
    Entry* entries = q.entries + (FAST ? (size_t)bin * q.cap : 0);
    const bool bs = q.baked_s != 0;
    const int baked = (bs || !q.baked_o) ? (int)bs : 1, half = (bs || !q.baked_o) ? q.half_s : q.half_o;

    // records (+ the reference's slice triples)
    for (int n = tid; n < q.N; n += PREP_CTA) {
        const float2 xy = reinterpret_cast<const float2*>(pts)[n];
        int win[12];
        recs[n] = make_rec(q, xy.x, xy.y, q.windows ? win : nullptr);
        if (q.windows) store_windows(q, bin, n, win);
    }
    if (tid == 0) band_base = 0;
    __syncthreads();

    for (int ty0 = 0; ty0 < q.tgy; ty0 += q.band_rows) {
        const int ty1 = min(ty0 + q.band_rows, q.tgy);
        const int nt = (ty1 - ty0) * q.tgx, t0 = ty0 * q.tgx;
        for (int i = tid; i < nt; i += PREP_CTA) cnt[i] = 0;
        __syncthreads();
        // 1. per-tile counts (each thread re-reads the records it wrote itself)
        for (int n = tid; n < q.N; n += PREP_CTA) {
            const PointRec r = recs[n];
            const int c_lo = r.uc & 0xffff, c_hi = r.uc >> 16, r_lo = r.ur & 0xffff, r_hi = r.ur >> 16;
            if (c_hi > c_lo && r_hi > r_lo) {
                const int ya = max(r_lo / q.th, ty0), yb = min((r_hi - 1) / q.th, ty1 - 1);
                for (int ty = ya; ty <= yb; ++ty)
                    for (int tx = c_lo / q.tw; tx <= (c_hi - 1) / q.tw; ++tx) atomicAdd(&cnt[(ty - ty0) * q.tgx + tx], 1);
            }
        }
        __syncthreads();
        // 2. exclusive scan over the band's tiles
        int beg, end;
        int run = block_exclusive_scan(cnt, nt, warp_tot, band_base, beg, end);
        for (int i = beg; i < end; ++i) {
            const int c = cnt[i];
            cnt[i] = run; cur[i] = run; tile_off[t0 + i] = run;
            run += c;
            if (FAST && c > WCH) q.ovf[1 + atomicAdd(q.ovf, 1)] = bin * q.T + t0 + i;
        }
        __syncthreads();
        if (tid == PREP_CTA - 1) band_base = run;      // the last thread's running total covers the whole band
        // 3. fill (arrival order)
        for (int n = tid; n < q.N; n += PREP_CTA) {
            const PointRec r = recs[n];
            const int c_lo = r.uc & 0xffff, c_hi = r.uc >> 16, r_lo = r.ur & 0xffff, r_hi = r.ur >> 16;
            if (c_hi > c_lo && r_hi > r_lo) {
                const int ya = max(r_lo / q.th, ty0), yb = min((r_hi - 1) / q.th, ty1 - 1);
                for (int ty = ya; ty <= yb; ++ty)
                    for (int tx = c_lo / q.tw; tx <= (c_hi - 1) / q.tw; ++tx) {
                        const int pos = atomicAdd(&cur[(ty - ty0) * q.tgx + tx], 1);
                        if (pos < q.cap) list[pos] = n;
                    }
            }
        }
        __syncthreads();
        // 4. order every tile's list by point index -> deterministic accumulation order
        for (int t = tid; t < nt; t += PREP_CTA) {
            const int b = cnt[t], e = min(cur[t], q.cap);
            if (FAST && e - b <= WCH) {
                // the common case: the whole list in registers (one load per element instead of one per comparison -- the
                // per-lane scattered re-reads were the kernel's L1 wavefront budget), sorted there, entries written in order
                int l[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) l[i] = (i < WCH && b + i < e) ? list[b + i] : 0x7fffffff;
                sort16(l);
#pragma unroll
                for (int i = 0; i < WCH; ++i) {
                    if (b + i < e) {
                        const PointRec& r = recs[l[i]];
                        store_entry(entries + b + i, r.p0, r.p1, r.ur, r.uc, (unsigned)l[i], baked, half);
                    }
                }
            } else if (FAST) {
                // rank sort straight into the entry list: independent loads, no serial chain through global memory
                for (int i = b; i < e; ++i) {
                    const int v = list[i];
                    int rank = 0;
                    for (int j = b; j < e; ++j) rank += list[j] < v;
                    const PointRec& r = recs[v];
                    store_entry(entries + b + rank, r.p0, r.p1, r.ur, r.uc, (unsigned)v, baked, half);
                }
            } else {
                for (int i = b + 1; i < e; ++i) {
                    const int v = list[i];
                    int j = i - 1;
                    while (j >= b && list[j] > v) { list[j + 1] = list[j]; --j; }
                    list[j + 1] = v;
                }
            }
        }
        __syncthreads();
    }
    if (tid == 0) tile_off[q.T] = band_base;
}

// One-pass binning for the warp-tile path (whole tile grid in one band, N <= 65535, everything below in shared memory).
// prepare_kernel<true> counts, scans, fills a global index list and then lets every thread sort and emit whole super tiles: two
// shared-memory atomics per (point, super tile) pair, and entry stores that scatter 32 x 16 bytes per instruction (profiles/r02x:
// lg_throttle + long scoreboard are two thirds of its stall samples).  Here
//   - a pair costs ONE atomic: the counter's old value is the point's slot in a fixed WCH-entry list per super tile (uint16 indices);
//   - the lists are sorted in registers in place (point order = deterministic accumulation order);
//   - the entries are written by whole warps, one super tile per step: lane (i, h) stores half h of entry i, so a store instruction
//     covers one contiguous run of <= 512 bytes.
// Super tiles with more than WCH candidates (clustered patterns; they go to the overflow kernels anyway) are completed by a second
// pass into the global index list; the first word of their (unused) slot row is the fill cursor.
struct Rec16 { float p0, p1; uint32_t ur, uc; };
// BANDED: the tile grid does not fit the shared arrays at once (textures beyond ~2048^2): the records are computed once, then the
// grid is binned in bands of q.band_rows tile rows, each with the same five phases.  !BANDED is the single-band kernel of config 3
// with the record computation merged into the slot pass.
// 48 registers: a resident CTA leaves a quarter of the register file to the CTAs of the scene randomisation, which runs next to it
template <bool BANDED>
__global__ void __maxnreg__(48) prepare_onepass_kernel(PrepParams q) {
    extern __shared__ __align__(16) int sm[];
    const int T = q.T;
    const int Tb = BANDED ? q.band_rows * q.tgx : T; // super tiles per band = capacity of the shared arrays
    int* cnt = sm;                                   // [Tb] candidates per super tile
    int* off = sm + Tb;                              // [Tb] exclusive offsets (into the sample's entry array)
    const int slot0 = (2 * Tb + 3) & ~3;             // 16-byte aligned rows
    unsigned short* slot = reinterpret_cast<unsigned short*>(sm + slot0);                         // [Tb][WCH]
    Rec16* recs = reinterpret_cast<Rec16*>(sm + slot0 + Tb * (WCH / 2));                           // [N]
    __shared__ int warp_tot[32];
    __shared__ int n_ovf, band_base;
    const int bin = blockIdx.x, tid = threadIdx.x;
    const float* pts = q.pts + (long long)bin * q.stride;
    int* tile_off = q.tile_off + (size_t)bin * (T + 1);
    int* list = q.list + (size_t)bin * q.cap;
    Entry* entries = q.entries + (size_t)bin * q.cap;
    const bool bs = q.baked_s != 0;
    const int baked = (bs || !q.baked_o) ? (int)bs : 1, half = (bs || !q.baked_o) ? q.half_s : q.half_o;
    auto record = [&](int n) {                       // the point's record (+ the reference's slice triples)
        const float2 xy = reinterpret_cast<const float2*>(pts)[n];
        int win[12];
        const PointRec rec = make_rec(q, xy.x, xy.y, q.windows ? win : nullptr);
        const Rec16 r = Rec16{rec.p0, rec.p1, rec.ur, rec.uc};
        recs[n] = r;
        if (q.windows) store_windows(q, bin, n, win);
        return r;
    };
    if (BANDED)
        for (int n = tid; n < q.N; n += PREP_CTA) record(n);
    if (tid == 0) band_base = 0;
    const int rows = BANDED ? q.band_rows : q.tgy;
#pragma unroll 1
    for (int ty0 = 0; ty0 < q.tgy; ty0 += rows) {
        const int ty1 = BANDED ? min(ty0 + rows, q.tgy) : q.tgy;
        const int nt = BANDED ? (ty1 - ty0) * q.tgx : T, t0 = ty0 * q.tgx;
        for (int i = tid; i < nt; i += PREP_CTA) cnt[i] = 0;
        if (tid == 0) n_ovf = 0;
        __syncthreads();
        // 1. (records +) slots
        for (int n = tid; n < q.N; n += PREP_CTA) {
            const Rec16 r = BANDED ? recs[n] : record(n);
            const int c_lo = r.uc & 0xffff, c_hi = r.uc >> 16, r_lo = r.ur & 0xffff, r_hi = r.ur >> 16;
            if (c_hi > c_lo && r_hi > r_lo) {
                int ya = r_lo / WT, yb = (r_hi - 1) / WT;                             // super tiles are 4 WT x WT texels (make_plan, fast path)
                if (BANDED) { ya = max(ya, ty0); yb = min(yb, ty1 - 1); }
                for (int ty = ya; ty <= yb; ++ty)
                    for (int tx = c_lo / (4 * WT); tx <= (c_hi - 1) / (4 * WT); ++tx) {
                        const int t = (ty - ty0) * q.tgx + tx;
                        const int pos = atomicAdd(&cnt[t], 1);
                        if (pos < WCH) slot[t * WCH + pos] = (unsigned short)n;
                    }
            }
        }
        __syncthreads();
        // 2. exclusive scan over the band's super tiles
        int beg, end;
        int run = block_exclusive_scan(cnt, nt, warp_tot, band_base, beg, end);
        for (int i = beg; i < end; ++i) {
            const int c = cnt[i];
            off[i] = run; tile_off[t0 + i] = run;
            run += c;
            if (c > WCH) {
                q.ovf[1 + atomicAdd(q.ovf, 1)] = bin * T + t0 + i;
                atomicAdd(&n_ovf, 1);
                *reinterpret_cast<int*>(slot + i * WCH) = 0;       // becomes the fill cursor of pass 3
            }
        }
        __syncthreads();
        if (tid == PREP_CTA - 1) band_base = run;                   // the last thread's running total covers the whole band
        // 3. overflow super tiles: the complete lists into the global list
        if (n_ovf > 0) {
            for (int n = tid; n < q.N; n += PREP_CTA) {
                const Rec16 r = recs[n];
                const int c_lo = r.uc & 0xffff, c_hi = r.uc >> 16, r_lo = r.ur & 0xffff, r_hi = r.ur >> 16;
                if (c_hi > c_lo && r_hi > r_lo) {
                    int ya = r_lo / WT, yb = (r_hi - 1) / WT;
                    if (BANDED) { ya = max(ya, ty0); yb = min(yb, ty1 - 1); }
                    for (int ty = ya; ty <= yb; ++ty)
                        for (int tx = c_lo / (4 * WT); tx <= (c_hi - 1) / (4 * WT); ++tx) {
                            const int t = (ty - ty0) * q.tgx + tx;
                            if (cnt[t] > WCH) {
                                const int pos = off[t] + atomicAdd(reinterpret_cast<int*>(slot + t * WCH), 1);
                                if (pos < q.cap) list[pos] = n;
                            }
                        }
                }
            }
            __syncthreads();
        }
        // 4. every super tile's list ordered by point index, in place; the overflow lists are ranked straight into their entries
        for (int t = tid; t < nt; t += PREP_CTA) {
            const int c = cnt[t], b = off[t];
            if (c > WCH) {
                const int e = min(b + c, q.cap);
                for (int i = b; i < e; ++i) {
                    const int v = list[i];
                    int rank = 0;
                    for (int j = b; j < e; ++j) rank += list[j] < v;
                    const Rec16 r = recs[v];
                    store_entry(entries + b + rank, r.p0, r.p1, r.ur, r.uc, (unsigned)v, baked, half);
                }
            } else if (c > 1) {
                uint4* row = reinterpret_cast<uint4*>(slot + t * WCH);
                const uint4 w0 = row[0], w1 = row[1];
                const unsigned w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
                int l[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) l[i] = i < c ? (int)((w[i >> 1] >> (16 * (i & 1))) & 0xffffu) : 0x7fffffff;
                sort16(l);
                unsigned o[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) o[i] = ((unsigned)l[2 * i] & 0xffffu) | ((unsigned)l[2 * i + 1] << 16);
                row[0] = make_uint4(o[0], o[1], o[2], o[3]);
                row[1] = make_uint4(o[4], o[5], o[6], o[7]);
            }
        }
        __syncthreads();
        // 5. entries: two super tiles per warp step, lane (hp, i) writes entry i of super tile t + hp --
        // 32 contiguous bytes per lane, one contiguous run per warp (consecutive super tiles are consecutive in the entry array)
        const int lane = tid & 31, wid = tid >> 5, i = lane & 15, hp = lane >> 4;
        const int tiles_per_warp = (((nt + 31) / 32) + 1) & ~1;
        const int tb = wid * tiles_per_warp, te = min(tb + tiles_per_warp, nt);
#pragma unroll 2
        for (int t = tb + hp; t < te; t += 2) {
            const int c = cnt[t], b = off[t];
            if (c <= WCH && i < c && b + i < q.cap) {
                const unsigned idx = slot[t * WCH + i];
                const Rec16 r = recs[idx];
                store_entry(entries + b + i, r.p0, r.p1, r.ur, r.uc, idx, baked, half);
            }
        }
        if (BANDED) __syncthreads();                               // the next band reuses the shared arrays
    }
    __syncthreads();
    if (tid == 0) tile_off[T] = band_base;
}

struct RasterParams {
    const PointRec* recs;
    const int* tile_off;
    const int* list;
    const Entry* entries;     // warp-tile kernels
    const int* ovf;           // [0] = overflow count, then the overflow super tiles
    const float* saved_softor;
    int shared_pattern;       // 1: every sample uses bin 0
    int N, ts0, ts1, tgx, tgy, T, cap;
    float sigma, rcp_sigma;
    float* out_sum; float* out_softor;            // forward
    const float* g_sum; const float* g_softor;    // backward
    float* d_pts;
    int eager;                // backward: request a super tile's first upstream boxes before its candidate list is known (dense patterns)
    int log_tgx, log_T;       // log2 of tgx and T when both are powers of two (item decode of the chunked backward by shifts), else -1
    float* loss;              // fused L1 backward: per-sample mean |softor - sum| (accumulated)
    float loss_inv;           // 1 / (ts0 * ts1)
};

__device__ __forceinline__ bool in_win(int v, uint32_t w) { return v >= (int)(w & 0xffff) && v < (int)(w >> 16); }

// g for one texel: identical operation order to the reference (rasterization.py:32-35):
// (dc*dc + dr*dr) / sigma, squared, negated, exp.
__device__ __forceinline__ float eval_g(float dx2, float dy, float sigma, float rcp_sigma, float& u) {
    const float d2 = __fadd_rn(dx2, __fmul_rn(dy, dy));
    u = div_by(d2, sigma, rcp_sigma);
    return exp_neg(__fmul_rn(u, u));
}

template <bool SUM, bool SOFTOR, bool SUM_T>
__global__ void __launch_bounds__(CTA) splat_fwd_kernel(RasterParams q) {
    __shared__ PointRec recs_s[CHUNK];
    const int tile = blockIdx.x % q.T, b = blockIdx.x / q.T;
    const int bin = q.shared_pattern ? 0 : b;
    const int tx = tile % q.tgx, ty = tile / q.tgx;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wc0 = tx * TW + (warp & 1) * 32, wr0 = ty * TH + (warp >> 1) * WROWS;
    const int c = wc0 + lane;
    const float cf = (float)c, rf0 = (float)wr0;
    const int* toff = q.tile_off + (size_t)bin * (q.T + 1);
    const int beg = toff[tile], end = toff[tile + 1];
    const int* list = q.list + (size_t)bin * q.cap;
    const PointRec* recs = q.recs + (size_t)bin * q.N;

    float acc_s[WROWS], acc_p[WROWS];
#pragma unroll
    for (int i = 0; i < WROWS; ++i) { acc_s[i] = 0.f; acc_p[i] = 1.f; }

    for (int base = beg; base < end; base += CHUNK) {
        const int n = min(CHUNK, end - base);
        __syncthreads();
        if (tid < n) recs_s[tid] = recs[list[base + tid]];
        __syncthreads();
        for (int k = 0; k < n; ++k) {
            const uint4 wa = reinterpret_cast<const uint4*>(&recs_s[k])[0];
            const uint4 wb = reinterpret_cast<const uint4*>(&recs_s[k])[1];
            const uint32_t uc = wb.z, ur = wb.w;
            // warp-uniform cull against this warp's 8x32 block
            if ((int)(uc >> 16) <= wc0 || (int)(uc & 0xffff) >= wc0 + 32 || (int)(ur >> 16) <= wr0 || (int)(ur & 0xffff) >= wr0 + WROWS) continue;
            const float p0 = __uint_as_float(wa.x), p1 = __uint_as_float(wa.y);
            const float dx = cf - p0;
            const float dx2 = __fmul_rn(dx, dx);
            const bool cs = SUM && in_win(c, wa.z), co = SOFTOR && in_win(c, wb.x);
            const int r_lo = ur & 0xffff, r_hi = ur >> 16;
#pragma unroll
            for (int i = 0; i < WROWS; ++i) {
                const int r = wr0 + i;
                if (r >= r_lo && r < r_hi) {                       // warp-uniform
                    float u;
                    const float g = eval_g(dx2, (rf0 + (float)i) - p1, q.sigma, q.rcp_sigma, u);
                    if (SUM) acc_s[i] += (cs && in_win(r, wa.w)) ? g : 0.f;
                    if (SOFTOR) acc_p[i] *= (co && in_win(r, wb.y)) ? (1.f - g) : 1.f;
                }
            }
        }
    }
    // epilogue: every texel of the tile is written exactly once
    const size_t frame = (size_t)q.ts0 * q.ts1;
    if (SOFTOR && c < q.ts0) {
        float* o = q.out_softor + (size_t)b * frame + c;
#pragma unroll
        for (int i = 0; i < WROWS; ++i)
            if (wr0 + i < q.ts1) o[(size_t)(wr0 + i) * q.ts0] = 1.f - acc_p[i];
    }
    if (SUM && c < q.ts0) {
        if (!SUM_T) {
            float* o = q.out_sum + (size_t)b * frame + c;
#pragma unroll
            for (int i = 0; i < WROWS; ++i)
                if (wr0 + i < q.ts1) o[(size_t)(wr0 + i) * q.ts0] = acc_s[i];
        } else {
            float* o = q.out_sum + (size_t)b * frame + (size_t)c * q.ts1 + wr0;   // [ts0, ts1]: 8 consecutive rows
            if ((q.ts1 & 3) == 0 && wr0 + WROWS <= q.ts1) {
                reinterpret_cast<float4*>(o)[0] = make_float4(acc_s[0], acc_s[1], acc_s[2], acc_s[3]);
                reinterpret_cast<float4*>(o)[1] = make_float4(acc_s[4], acc_s[5], acc_s[6], acc_s[7]);
            } else {
#pragma unroll
                for (int i = 0; i < WROWS; ++i)
                    if (wr0 + i < q.ts1) o[i] = acc_s[i];
            }
        }
    }
}

template <bool SUM, bool SOFTOR, bool SUM_T>
__global__ void __launch_bounds__(CTA) splat_bwd_kernel(RasterParams q) {
    __shared__ PointRec recs_s[CHUNK];
    __shared__ float dp_s[CHUNK][2];
    extern __shared__ float gcache[];      // SOFTOR: [8 warps][KCACHE][8 rows][32 lanes]
    const int tile = blockIdx.x % q.T, b = blockIdx.x / q.T;
    const int bin = q.shared_pattern ? 0 : b;
    const int tx = tile % q.tgx, ty = tile / q.tgx;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wc0 = tx * TW + (warp & 1) * 32, wr0 = ty * TH + (warp >> 1) * WROWS;
    const int c = wc0 + lane;
    const float cf = (float)c, rf0 = (float)wr0;
    const int* toff = q.tile_off + (size_t)bin * (q.T + 1);
    const int beg = toff[tile], end = toff[tile + 1];
    if (beg == end) return;
    const int* list = q.list + (size_t)bin * q.cap;
    const PointRec* recs = q.recs + (size_t)bin * q.N;
    const size_t frame = (size_t)q.ts0 * q.ts1;
    float* gc = gcache + (SOFTOR ? warp * KCACHE * WROWS * 32 + lane : 0);

    // upstream gradients of this lane's 8 texels
    float gs[WROWS], go[WROWS];
#pragma unroll
    for (int i = 0; i < WROWS; ++i) { gs[i] = 0.f; go[i] = 0.f; }
    if (c < q.ts0) {
        if (SOFTOR) {
            const float* p = q.g_softor + (size_t)b * frame + c;
#pragma unroll
            for (int i = 0; i < WROWS; ++i)
                if (wr0 + i < q.ts1) go[i] = __ldg(p + (size_t)(wr0 + i) * q.ts0);
        }
        if (SUM) {
            if (!SUM_T) {
                const float* p = q.g_sum + (size_t)b * frame + c;
#pragma unroll
                for (int i = 0; i < WROWS; ++i)
                    if (wr0 + i < q.ts1) gs[i] = __ldg(p + (size_t)(wr0 + i) * q.ts0);
            } else {
                const float* p = q.g_sum + (size_t)b * frame + (size_t)c * q.ts1 + wr0;
                if ((q.ts1 & 3) == 0 && wr0 + WROWS <= q.ts1) {
                    const float4 a = __ldg(reinterpret_cast<const float4*>(p));
                    const float4 d = __ldg(reinterpret_cast<const float4*>(p) + 1);
                    gs[0] = a.x; gs[1] = a.y; gs[2] = a.z; gs[3] = a.w; gs[4] = d.x; gs[5] = d.y; gs[6] = d.z; gs[7] = d.w;
                } else {
#pragma unroll
                    for (int i = 0; i < WROWS; ++i)
                        if (wr0 + i < q.ts1) gs[i] = __ldg(p + i);
                }
            }
        }
    }

    // ---- pass 1: product of the non-zero (1-g) factors per texel + zero bookkeeping, g cached ----
    float prod[WROWS];
    uint32_t z1 = 0, z2 = 0;      // bit i: >=1 / >=2 exact-zero factors at row i
#pragma unroll
    for (int i = 0; i < WROWS; ++i) prod[i] = 1.f;
    if (SOFTOR) {
        int kk = 0;               // warp-uniform index of the next relevant candidate
        for (int base = beg; base < end; base += CHUNK) {
            const int n = min(CHUNK, end - base);
            __syncthreads();
            if (tid < n) recs_s[tid] = recs[list[base + tid]];
            __syncthreads();
            for (int k = 0; k < n; ++k) {
                const uint4 wa = reinterpret_cast<const uint4*>(&recs_s[k])[0];
                const uint4 wb = reinterpret_cast<const uint4*>(&recs_s[k])[1];
                const uint32_t uc = wb.z, ur = wb.w;
                if ((int)(uc >> 16) <= wc0 || (int)(uc & 0xffff) >= wc0 + 32 || (int)(ur >> 16) <= wr0 || (int)(ur & 0xffff) >= wr0 + WROWS) continue;
                const float p0 = __uint_as_float(wa.x), p1 = __uint_as_float(wa.y);
                const float dx = cf - p0;
                const float dx2 = __fmul_rn(dx, dx);
                const bool co = in_win(c, wb.x);
                const int r_lo = ur & 0xffff, r_hi = ur >> 16;
#pragma unroll
                for (int i = 0; i < WROWS; ++i) {
                    const int r = wr0 + i;
                    if (r >= r_lo && r < r_hi) {
                        float u;
                        const float g = eval_g(dx2, (rf0 + (float)i) - p1, q.sigma, q.rcp_sigma, u);
                        if (kk < KCACHE) gc[(kk * WROWS + i) * 32] = g;
                        if (co && in_win(r, wb.y)) {
                            const float om = 1.f - g;
                            if (om == 0.f) { z2 |= z1 & (1u << i); z1 |= 1u << i; }
                            else prod[i] *= om;
                        }
                    }
                }
                ++kk;
            }
        }
    }

    // ---- pass 2: dL/dg per (texel, point) -> d/dp, reduced over the tile ----
    const float k0 = 4.f * (float)q.ts0 * q.rcp_sigma, k1 = 4.f * (float)q.ts1 * q.rcp_sigma;
    int kk = 0;
    for (int base = beg; base < end; base += CHUNK) {
        const int n = min(CHUNK, end - base);
        if (!SOFTOR || end - beg > CHUNK) {      // single-chunk soft-OR tiles still hold their records
            __syncthreads();
            if (tid < n) recs_s[tid] = recs[list[base + tid]];
        }
        if (tid < n) { dp_s[tid][0] = 0.f; dp_s[tid][1] = 0.f; }
        __syncthreads();
        for (int k = 0; k < n; ++k) {
            const uint4 wa = reinterpret_cast<const uint4*>(&recs_s[k])[0];
            const uint4 wb = reinterpret_cast<const uint4*>(&recs_s[k])[1];
            const uint32_t uc = wb.z, ur = wb.w;
            if ((int)(uc >> 16) <= wc0 || (int)(uc & 0xffff) >= wc0 + 32 || (int)(ur >> 16) <= wr0 || (int)(ur & 0xffff) >= wr0 + WROWS) continue;
            const float p0 = __uint_as_float(wa.x), p1 = __uint_as_float(wa.y);
            const float dx = cf - p0;
            const float dx2 = __fmul_rn(dx, dx);
            const bool cs = SUM && in_win(c, wa.z), co = SOFTOR && in_win(c, wb.x);
            const int r_lo = ur & 0xffff, r_hi = ur >> 16;
            float a0 = 0.f, a1 = 0.f;
#pragma unroll
            for (int i = 0; i < WROWS; ++i) {
                const int r = wr0 + i;
                if (r >= r_lo && r < r_hi) {
                    const float dy = (rf0 + (float)i) - p1;
                    float u, g;
                    if (SOFTOR && kk < KCACHE) {
                        g = gc[(kk * WROWS + i) * 32];
                        u = __fadd_rn(dx2, __fmul_rn(dy, dy)) * q.rcp_sigma;
                    } else {
                        g = eval_g(dx2, dy, q.sigma, q.rcp_sigma, u);
                    }
                    float coef = 0.f;
                    if (SUM && cs && in_win(r, wa.w)) coef = gs[i];
                    if (SOFTOR && co && in_win(r, wb.y)) {
                        const float om = 1.f - g;
                        float excl;                                   // prod_{m != n} (1 - g_m)
                        if (!(z1 & (1u << i))) excl = __fdividef(prod[i], om);
                        else excl = (om == 0.f && !(z2 & (1u << i))) ? prod[i] : 0.f;
                        coef = fmaf(go[i], excl, coef);
                    }
                    const float w = coef * g * u;
                    a0 = fmaf(w, dx, a0);
                    a1 = fmaf(w, dy, a1);
                }
            }
            a0 = warp_sum(a0);
            a1 = warp_sum(a1);
            if (lane == 0) { atomicAdd(&dp_s[k][0], a0); atomicAdd(&dp_s[k][1], a1); }
            ++kk;
        }
        __syncthreads();
        if (tid < n) {
            float* o = q.d_pts + ((size_t)b * q.N + list[base + tid]) * 2;
            const float v0 = dp_s[tid][0] * k0, v1 = dp_s[tid][1] * k1;
            if (v0 != 0.f) atomicAdd(o, v0);
            if (v1 != 0.f) atomicAdd(o + 1, v1);
        }
    }
}

#include "ffb_splat_wt.cuh"
#include "ffb_splat_st.cuh"

static WtConsts wt_consts(const ffb_splat_desc* d, const Plan& p) {
    WtConsts fc;
    fc.K2 = (float)(-1.4426950408889634 / ((double)d->sigma * (double)d->sigma));
    fc.thr_s = 4.f * (float)p.H_s + 2.f;
    fc.thr_o = 4.f * (float)p.H_o + 2.f;
    fc.hs = (float)p.H_s + 0.5f;
    fc.ho = (float)p.H_o + 0.5f;
    fc.c1 = 1.00000011920928955078125f;      // 1 + 2^-23
    // backward tile culling: a tile whose nearest texel centre has g < 1e-7 is skipped.  Measured at config 3 against fp64
    // (scripts/grad_precision.py): error relative to the gradient norm 5.2e-7 at 1e-7 and 5.3e-7 at 1e-9 (the
    // round-1 threshold) -- below the kernels' own rounding -- and 8.2e-7 at 1e-6; 7 % fewer (candidate, tile) visits than at 1e-9.
    // Worst case (upstream of one sign, dropped ring all on one side): 170 texels x 3.5e-7 against one-sided sums of ~20, 1e-5 of a
    // non-cancelling gradient's norm = a tenth of the parity tolerance.
    fc.disc2 = (float)((double)d->sigma * sqrt(16.11809565095832));       // (d2 / sigma)^2 = ln(1e7)
    fc.disc2_f = (float)((double)d->sigma * sqrt(17.5) * 1.02);           // same margin as the exact soft-OR no-op radius h_o (make_plan)
    fc.near2 = (float)((double)d->sigma * sqrt(5.545177444479562));       // (d2 / sigma)^2 = ln(2^8)
    fc.s2 = (float)(sqrt(1.4426950408889634) / (double)d->sigma);
    fc.rs2 = (float)((double)d->sigma / sqrt(1.4426950408889634));
    {
        const double s2 = sqrt(1.4426950408889634) / (double)d->sigma, r1 = sqrt(s2);
        fc.r1 = (float)r1;
        fc.rs3 = (float)(1.0 / (s2 * r1));
        fc.hs_r = (float)(((double)p.H_s + 0.5) * r1);
        fc.m_r = (float)(-4.0 / r1);
        fc.thr_r = 4.f * (float)p.H_s + 2.f;
    }
    return fc;
}
// main kernel over the strip grid, then the overflow kernel over its (normally empty) list
template <typename K, typename KO>
static int launch_wt(K kernel, KO overflow, const RasterParams& q, const WtConsts& fc, const OvfParams& o, int B, cudaStream_t st,
                     int cta = WT_CTA, size_t smem = 0, size_t smem_ovf = 0) {
    const int warps = cta / 32;
    const unsigned gy = (unsigned)((q.tgy + warps * WT_S - 1) / (warps * WT_S));
    if (B > 65535 || gy > 65535) return fail_arg(FFB_E_LIMIT, "splat: B or the tile rows exceed the grid limit (65535)");
    if (smem > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (smem_ovf > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(overflow, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ovf));
    kernel<<<dim3((unsigned)q.tgx, gy, (unsigned)B), cta, smem, st>>>(q, fc);
    FFB_CUDA(cudaGetLastError());
    overflow<<<kNumSMs, WT_CTA, smem_ovf, st>>>(q, fc, o);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

// TMA-store forward over the strip grid (tensor maps of the outputs as kernel parameters)
template <typename K, typename KO>
static int launch_fwd_tma(K kernel, KO overflow, const RasterParams& q, const WtConsts& fc, const OvfParams& o, int B, cudaStream_t st,
                          const CUtensorMap& ms, const CUtensorMap& mo, size_t stage_bytes) {
    const unsigned gy = (unsigned)((q.tgy + WF_WARPS * WF_S - 1) / (WF_WARPS * WF_S));
    if (B > 65535 || gy > 65535) return fail_arg(FFB_E_LIMIT, "splat: B or the tile rows exceed the grid limit (65535)");
    const size_t smem = (size_t)WF_WARPS * (2 * TMA_TILE_BYTES + stage_bytes);
    if (smem > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<dim3((unsigned)q.tgx, gy, (unsigned)B), WF_CTA, smem, st>>>(q, fc, ms, mo);
    FFB_CUDA(cudaGetLastError());
    overflow<<<kNumSMs, WT_CTA, 0, st>>>(q, fc, o);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

// tensor maps of the upstream arrays (kernel parameters of the TMA-fed backward kernels)
struct BwdMaps {
    CUtensorMap gs, go, sv, ot;
};
// TMA-fed backward over the same strip grid
template <typename K, typename KO>
static int launch_bwd_tma(K kernel, KO overflow, const RasterParams& q, const WtConsts& fc, const OvfParams& o, int B, cudaStream_t st,
                          const BwdMaps& m, size_t stage_bytes, size_t smem_ovf) {
    const unsigned gy = (unsigned)((q.tgy + WB_WARPS * WT_S - 1) / (WB_WARPS * WT_S));
    if (B > 65535 || gy > 65535) return fail_arg(FFB_E_LIMIT, "splat: B or the tile rows exceed the grid limit (65535)");
    const size_t smem = (size_t)WB_WARPS * 3 * TMA_TILE_BYTES + 64 + stage_bytes * WB_WARPS;
    if (smem > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (smem_ovf > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(overflow, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ovf));
    kernel<<<dim3((unsigned)q.tgx, gy, (unsigned)B), WB_CTA, smem, st>>>(q, fc, m.gs, m.go, m.sv);
    FFB_CUDA(cudaGetLastError());
    overflow<<<kNumSMs, WT_CTA, smem_ovf, st>>>(q, fc, o);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

__device__ unsigned st_counters[64];      // work counters of the loss-mode backward launches in flight (ffb_splat_st.cuh)

// One zeroed counter per launch: a slot of the per-device pool, handed out round-robin across ALL instantiations and streams (64
// launches may be in flight; a launch lasts milliseconds), zeroed on the launching stream.
static int st_counter_slot(cudaStream_t st, unsigned** counter) {
    static unsigned* pool[64] = {nullptr};
    static unsigned turn = 0;
    int dev = 0;
    FFB_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return fail_arg(FFB_E_LIMIT, "splat: device ordinal >= 64");
    if (!pool[dev]) FFB_CUDA(cudaGetSymbolAddress(reinterpret_cast<void**>(&pool[dev]), st_counters));
    *counter = pool[dev] + (__atomic_fetch_add(&turn, 1u, __ATOMIC_RELAXED) & 63u);
    FFB_CUDA(cudaMemsetAsync(*counter, 0, sizeof(unsigned), st));
    return 0;
}

// super-tile backward (ffb_splat_st.cuh) for dense patterns (q.eager), then the overflow kernel; splat_bwd_stp's item loop with the
// two-stage request pipeline.
//   chunk > 0 (plain mode, 8): a one-warp CTA walks `chunk` consecutive (super tile, sample) items; the hardware block scheduler
//     balances the 131 k CTAs of a config-3 launch.  1.91 ms per 256 samples inside the bench step against 2.05 for the one-shot form
//     (whose warp slots stay empty ~2 of every ~9 us) and 2.6-2.7 for the counter form (profiles/r02x/forms.log);
//   chunk == 0 (loss mode): 148 x 22 resident warps claim items from a global counter.  The fused L1 step measured 4.03 ms end to end
//     against 4.07 with chunks of 4 and 4.18 with chunks of 8 (B200 at 1000 W, 5 alternating rounds of bench.py --steps 20).
template <typename K, typename KO>
static int launch_bwd_stp(K kernel, KO overflow, const RasterParams& q, const WtConsts& fc, const OvfParams& o, int B, cudaStream_t st,
                          const BwdMaps& m, size_t smem, size_t smem_ovf, int chunk) {
    if (B > 65535 || q.tgy > 65535) return fail_arg(FFB_E_LIMIT, "splat: B or the tile rows exceed the grid limit (65535)");
    const long long items = (long long)q.T * B;
    if (items > 0x7fff0000LL) return fail_arg(FFB_E_LIMIT, "splat: 2^31 (super tile, sample) items or more in one backward");
    if (smem_ovf > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(overflow, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ovf));
    static int occ = 0;                                     // per instantiation (the function is a template): queried on every call, the fused L1 step ran 4.15-4.27 ms end to end instead of 4.01-4.05
    if (occ == 0) {
        if (smem > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        FFB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        // queried with the size rounded up to the next KB, which stands in for the 1 KB the system reserves per CTA: with the exact size
        // the query reported more CTAs per SM than ncu showed resident (profiles/r02z/ncu_loss_summary.txt), and 148 CTAs of the counter
        // form started only when the others were done
        FFB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, 32, (smem + 1023) & ~(size_t)1023));
        if (occ < 1) occ = 1;
    }
    unsigned* counter = nullptr;
    long long grid = chunk > 0 ? (items + chunk - 1) / chunk : 0;
    if (chunk == 0) {
        if (int rc = st_counter_slot(st, &counter)) return rc;
        // 22 resident warps per SM: 2.31 / 2.26 / 2.22 ms per 256 samples with 19 / 20 / 22
        grid = (long long)kNumSMs * (occ < 22 ? occ : 22);
        if (grid > items) grid = items;
    }
    kernel<<<(unsigned)grid, 32, smem, st>>>(q, fc, m.gs, m.go, m.sv, m.ot, (int)items, counter, chunk);
    FFB_CUDA(cudaGetLastError());
    overflow<<<kNumSMs, WT_CTA, smem_ovf, st>>>(q, fc, o);
    FFB_CUDA(cudaGetLastError());
    return 0;
}
// super-tile backward for sparse patterns: one one-warp CTA of splat_bwd_st per (super tile, sample), then the overflow kernel
template <typename K, typename KO>
static int launch_bwd_st(K kernel, KO overflow, const RasterParams& q, const WtConsts& fc, const OvfParams& o, int B, cudaStream_t st,
                         const BwdMaps& m, size_t smem, size_t smem_ovf) {
    if (B > 65535 || q.tgy > 65535) return fail_arg(FFB_E_LIMIT, "splat: B or the tile rows exceed the grid limit (65535)");
    if (smem > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (smem_ovf > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(overflow, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ovf));
    kernel<<<dim3((unsigned)q.tgx, (unsigned)q.tgy, (unsigned)B), 32, smem, st>>>(q, fc, m.gs, m.go);
    FFB_CUDA(cudaGetLastError());
    overflow<<<kNumSMs, WT_CTA, smem_ovf, st>>>(q, fc, o);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

template <typename K>
static int launch_raster(K kernel, const RasterParams& q, int B, cudaStream_t st, size_t smem = 0) {
    const long long grid = (long long)B * q.T;
    if (grid > 0x7fffffffLL) return fail_arg(FFB_E_LIMIT, "splat: B * tiles exceeds the grid limit");
    // static + dynamic shared memory may exceed the 48 KB default even when the dynamic part alone does not
    if (smem > 32 * 1024) FFB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<(unsigned)grid, CTA, smem, st>>>(q);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

static void fill_raster(const ffb_splat_desc* d, const Plan& p, const void* ws, RasterParams& q) {
    const char* w = reinterpret_cast<const char*>(ws);
    q.recs = reinterpret_cast<const PointRec*>(w + p.off_recs);
    q.tile_off = reinterpret_cast<const int*>(w + p.off_tileoff);
    q.list = reinterpret_cast<const int*>(w + p.off_list);
    q.entries = reinterpret_cast<const Entry*>(w + p.off_entries);
    q.ovf = reinterpret_cast<const int*>(w + p.off_ovf);
    q.saved_softor = nullptr;
    q.shared_pattern = d->pts_batch_stride == 0;
    q.N = d->N; q.ts0 = d->ts0; q.ts1 = d->ts1; q.tgx = p.tgx; q.tgy = p.tgy; q.T = p.T; q.cap = p.cap;
    q.sigma = d->sigma; q.rcp_sigma = 1.0f / d->sigma;
    q.out_sum = nullptr; q.out_softor = nullptr; q.g_sum = nullptr; q.g_softor = nullptr; q.d_pts = nullptr;
    q.loss = nullptr; q.loss_inv = 0.f;
    {
        // expected candidates per 64x16 super tile for points spread over the texture: above ~2 nearly every super tile has work
        const double wwin = 2.0 * (p.H_s > p.H_o ? p.H_s : p.H_o) + 1.0;
        const double per_tile = (double)d->N * (wwin + 4 * WT - 1) * (wwin + WT - 1) / ((double)d->ts0 * (double)d->ts1);
        const char* e = getenv("FFB_SPLAT_EAGER");
        q.eager = e ? (e[0] == '1') : (per_tile >= 2.0);
        auto lg = [](int v) { int l = 0; while ((1 << l) < v) ++l; return (1 << l) == v ? l : -1; };
        q.log_tgx = lg(p.tgx); q.log_T = lg(p.T);
        if (q.log_tgx < 0 || q.log_T < 0) q.log_tgx = q.log_T = -1;
    }
}

// ---- dense API-compat kernels -----------------------------------------------------------------------
// sx, sy: the scale applied to the points (texture_size for rasterize_points, 1 for rasterize_points_in_non_ndc)
__global__ void __launch_bounds__(256) dense_fwd_kernel(const float* __restrict__ pts, int N, int ts0, int ts1, float sx, float sy, float sigma,
                                                        float rcp_sigma, float* __restrict__ out) {
    const size_t frame = (size_t)ts0 * ts1;
    const size_t total = frame * N;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int n = (int)(i / frame);
        const size_t t = i - (size_t)n * frame;
        const int r = (int)(t / ts0), c = (int)(t - (size_t)r * ts0);
        const float dx = (float)c - pts[2 * n] * sx;
        const float dy = (float)r - pts[2 * n + 1] * sy;
        const float d2 = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
        const float u = div_by(d2, sigma, rcp_sigma);
        const float w = __fmul_rn(u, u);
        out[i] = w > 87.f ? 0.f : exp_neg(w);
    }
}

__global__ void __launch_bounds__(256) dense_bwd_kernel(const float* __restrict__ pts, int N, int ts0, int ts1, float sx, float sy, float sigma,
                                                        float rcp_sigma, const float* __restrict__ g_out, float* __restrict__ d_pts) {
    // grid = (chunks, N): each CTA reduces a slice of one point's frame
    const int n = blockIdx.y;
    const size_t frame = (size_t)ts0 * ts1;
    const float p0 = pts[2 * n] * sx, p1 = pts[2 * n + 1] * sy;
    const float* go = g_out + (size_t)n * frame;
    float a0 = 0.f, a1 = 0.f;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < frame; t += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(t / ts0), c = (int)(t - (size_t)r * ts0);
        const float dx = (float)c - p0, dy = (float)r - p1;
        const float u = (dx * dx + dy * dy) * rcp_sigma;
        const float w = u * u;
        if (w <= 87.f) {
            const float q = go[t] * exp_neg(w) * u;
            a0 = fmaf(q, dx, a0);
            a1 = fmaf(q, dy, a1);
        }
    }
    __shared__ float red[2][8];
    a0 = warp_sum(a0); a1 = warp_sum(a1);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a0; red[1][threadIdx.x >> 5] = a1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float s0 = 0.f, s1 = 0.f;
        for (int i = 0; i < 8; ++i) { s0 += red[0][i]; s1 += red[1][i]; }
        atomicAdd(&d_pts[2 * n], s0 * 4.f * sx * rcp_sigma);
        atomicAdd(&d_pts[2 * n + 1], s1 * 4.f * sy * rcp_sigma);
    }
}

// out[j] = sum_b in[b, j] in a fixed order (deterministic): 32 columns per CTA, the samples split over 8 warps (each
// walks its contiguous share with four loads in flight), partial sums folded in warp order
__global__ void __launch_bounds__(256) reduce_samples_kernel(const float* __restrict__ in, int B, long long row, float* __restrict__ out) {
    __shared__ float part[8][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long j = (long long)blockIdx.x * 32 + lane;
    const int per = (B + 7) / 8, b0 = w * per, b1 = min(b0 + per, B);
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    if (j < row) {
        int b = b0;
        for (; b + 3 < b1; b += 4) {
            s0 += in[(long long)b * row + j]; s1 += in[(long long)(b + 1) * row + j];
            s2 += in[(long long)(b + 2) * row + j]; s3 += in[(long long)(b + 3) * row + j];
        }
        for (; b < b1; ++b) s0 += in[(long long)b * row + j];
    }
    part[w][lane] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (w == 0 && j < row) {
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += part[k][lane];
        out[j] = s;
    }
}

// texture-sized rows (shared-pattern backward: upstream gradients summed over the samples).  out[g, j] = sum of the (up to)
// 8 samples of group g: warp w of a CTA reads sample 8 g + w, a lane owns four float4 columns (four 512-byte warp accesses
// in flight), the eight partial rows are folded through shared memory in warp order.  The grid walks the column blocks of
// one group before the next group, so the CTAs in flight touch 8 sample planes at a time: a first version that let every
// CTA walk all B planes (256 x 16.8 MB apart) ran at 0.45 TB/s -- TLB reach -- instead of streaming speed.
__global__ void __launch_bounds__(256) reduce_groups_kernel(const float4* __restrict__ in, int B, long long row4, float4* __restrict__ out) {
    __shared__ float4 part[8][4][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, g = blockIdx.y;
    const long long j0 = (long long)blockIdx.x * 128 + lane;
    const int b = 8 * g + w;
    float4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const long long j = j0 + 32 * k;
        v[k] = (b < B && j < row4) ? __ldcs(in + (long long)b * row4 + j) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) part[w][k][lane] = v[k];
    __syncthreads();
    if (w < 4) {                                   // warp k folds column quad k
        const long long j = j0 + 32 * w;
        if (j < row4) {
            float4 s = part[0][w][lane];
#pragma unroll
            for (int q = 1; q < 8; ++q) { const float4 t = part[q][w][lane]; s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w; }
            out[(long long)g * row4 + j] = s;
        }
    }
}

// Fold over this rank's samples + one-shot all-reduce over NVLink peer memory, one kernel (SURVEY.md 8(e): the path's only
// exchange, [N,2] floats per step).  A CTA folds 32 columns over the B samples like reduce_samples_kernel, PUSHES its 32
// partial sums into slot [rank] of every peer's receive buffer (plain stores through the NVSwitch fabric), publishes them
// with a system-scope fence and a per-(rank, CTA) flag written into every peer's flag array, waits until the flags of all
// ranks for this CTA show the current epoch, then sums the `world` slots of its own buffer in rank order -- every rank adds
// in the same order, so the result is bit-identical everywhere.  No grid-wide barrier: CTA c only depends on CTA c of the
// peers, and all CTAs of the launch are resident.  Receive buffers are double buffered by epoch parity; the flags only grow.
struct PeerTable {
    float* recv[8];             // per rank: [2][world][row] receive slots (symmetric memory)
    unsigned* flag[8];          // per rank: [world][n_cta] epochs
};
__global__ void __launch_bounds__(256) fold_allreduce_kernel(const float* __restrict__ in, int B, long long row, PeerTable pt, int rank, int world,
                                                             unsigned epoch, float* __restrict__ out, int* __restrict__ err) {
    __shared__ float part[8][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long j = (long long)blockIdx.x * 32 + lane;
    const int per = (B + 7) / 8, b0 = w * per, b1 = min(b0 + per, B);
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    if (j < row) {
        int b = b0;
        for (; b + 3 < b1; b += 4) {
            s0 += in[(long long)b * row + j]; s1 += in[(long long)(b + 1) * row + j];
            s2 += in[(long long)(b + 2) * row + j]; s3 += in[(long long)(b + 3) * row + j];
        }
        for (; b < b1; ++b) s0 += in[(long long)b * row + j];
    }
    part[w][lane] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (w != 0) return;
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += part[k][lane];
    const size_t slot = ((size_t)(epoch & 1u) * world + rank) * row;
    if (j < row)
        for (int r = 0; r < world; ++r) pt.recv[r][slot + j] = s;                 // push: remote stores
    __threadfence_system();
    __syncwarp();
    if (lane < world) {
        unsigned* f = pt.flag[lane] + (size_t)rank * gridDim.x + blockIdx.x;       // my flag in peer `lane`'s array
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(epoch) : "memory");
        const unsigned* mine = pt.flag[rank] + (size_t)lane * gridDim.x + blockIdx.x;   // peer `lane`'s flag in my array
        unsigned v = 0;
        long long spins = 0;
        do {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
        } while ((int)(v - epoch) < 0 && ++spins < (1ll << 26));
        if ((int)(v - epoch) < 0) atomicExch(err, 1);                              // a peer never arrived: report instead of hanging
    }
    __syncwarp();
    if (j < row) {
        const float* mybuf = pt.recv[rank] + (size_t)(epoch & 1u) * world * row;
        float t = 0.f;
        for (int r = 0; r < world; ++r) t += __ldcv(mybuf + (size_t)r * row + j);
        out[j] = t;
    }
}

// mean |a - b| per sample and its gradients.  grid = (row blocks, B); each CTA handles 32x32 texels so the
// transposed operand is read/written through a shared-memory transpose.
template <bool BT>
__global__ void __launch_bounds__(256) l1_kernel(const float* __restrict__ a, const float* __restrict__ bsrc, int ts0, int ts1,
                                                 float inv_numel, float* __restrict__ loss, float* __restrict__ ga, float* __restrict__ gb) {
    __shared__ float tile[32][33];
    __shared__ float red[8];
    const int tiles_x = (ts0 + 31) / 32;
    const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
    const int smp = blockIdx.y;
    const size_t frame = (size_t)ts0 * ts1;
    const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;      // 32 x 8 threads
    const float* A = a + (size_t)smp * frame;
    const float* Bm = bsrc + (size_t)smp * frame;
    float part = 0.f;
    if (BT) {   // stage b^T tile: b is [ts0, ts1]; element (r,c) of the natural frame lives at b[c*ts1 + r]
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int cc = tx * 32 + ly + j * 8, rr = ty * 32 + lx;
            tile[ly + j * 8][lx] = (cc < ts0 && rr < ts1) ? Bm[(size_t)cc * ts1 + rr] : 0.f;
        }
        __syncthreads();
    }
    float sgn[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int r = ty * 32 + ly + j * 8, c = tx * 32 + lx;
        sgn[j] = 0.f;
        if (r < ts1 && c < ts0) {
            const float av = A[(size_t)r * ts0 + c];
            const float bv = BT ? tile[lx][ly + j * 8] : Bm[(size_t)r * ts0 + c];
            const float d = av - bv;
            part += fabsf(d);
            sgn[j] = d > 0.f ? inv_numel : (d < 0.f ? -inv_numel : 0.f);
            if (ga) ga[(size_t)smp * frame + (size_t)r * ts0 + c] = sgn[j];
            if (gb && !BT) gb[(size_t)smp * frame + (size_t)r * ts0 + c] = -sgn[j];
        }
    }
    if (BT && gb) {
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) tile[lx][ly + j * 8] = -sgn[j];
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int cc = tx * 32 + ly + j * 8, rr = ty * 32 + lx;
            if (cc < ts0 && rr < ts1) gb[(size_t)smp * frame + (size_t)cc * ts1 + rr] = tile[ly + j * 8][lx];
        }
    }
    part = warp_sum(part);
    if (lx == 0) red[ly] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
        for (int i = 0; i < 8; ++i) s += red[i];
        atomicAdd(&loss[smp], s * inv_numel);
    }
}

}  // namespace splat
}  // namespace ffb

using namespace ffb;
using namespace ffb::splat;

extern "C" size_t ffb_splat_workspace_bytes(const ffb_splat_desc* d) {
    Plan p;
    if (make_plan(d, &p)) return 0;
    return p.total;
}

extern "C" int ffb_splat_prepare(const ffb_splat_desc* d, const float* pts, void* workspace, size_t workspace_bytes,
                                 int32_t* windows_out, void* stream) {
    Plan p;
    if (int rc = make_plan(d, &p)) return rc;
    if (!pts || !workspace) return fail_arg(FFB_E_ARG, "splat_prepare: null pointer");
    if (workspace_bytes < p.total) return fail_arg(FFB_E_WORKSPACE, "splat_prepare: workspace too small");
    char* w = reinterpret_cast<char*>(workspace);
    PrepParams q;
    q.pts = pts; q.stride = d->pts_batch_stride;
    q.N = d->N; q.ts0 = d->ts0; q.ts1 = d->ts1; q.tgx = p.tgx; q.tgy = p.tgy; q.T = p.T; q.cap = p.cap;
    q.tw = p.tw; q.th = p.th; q.band_rows = p.band_rows;
    q.baked_s = d->num_std_sum > 0; q.fp_s = p.fp_s; q.half_s = p.half_s; q.h_s = p.h_s;
    q.baked_o = d->num_std_softor > 0; q.fp_o = p.fp_o; q.half_o = p.half_o; q.h_o = p.h_o;
    q.h_union = p.H_s > p.H_o ? p.H_s : p.H_o;
    q.recs = reinterpret_cast<PointRec*>(w + p.off_recs);
    q.tile_off = reinterpret_cast<int*>(w + p.off_tileoff);
    q.list = reinterpret_cast<int*>(w + p.off_list);
    q.entries = reinterpret_cast<Entry*>(w + p.off_entries);
    q.ovf = reinterpret_cast<int*>(w + p.off_ovf);
    q.windows = windows_out;
    const size_t smem = (size_t)p.band_rows * p.tgx * 2 * sizeof(int);
    if (p.fast) {
        FFB_CUDA(cudaMemsetAsync(q.ovf, 0, sizeof(int), as_stream(stream)));
        // one-pass binning (uint16 slots, so N <= 65535): whole grid at once when it fits (config 3: 4096 super tiles + 4096
        // records = 224 KB), otherwise in bands of tile rows.  When not even one tile row fits (about 14,400 points), count / scan /
        // fill with the records in the workspace.
        auto smem_for = [&](int rows) {
            const size_t tiles = (size_t)rows * p.tgx;
            return ((tiles * 2 + 3) & ~(size_t)3) * sizeof(int) + tiles * WCH * sizeof(unsigned short) + (size_t)d->N * sizeof(Rec16);
        };
        const size_t budget = 226 * 1024;
        if (d->N <= 65535 && smem_for(1) <= budget) {
            const char* eb = getenv("FFB_PREP_BAND_ROWS");      // tests: bin in bands of this many tile rows (at most what fits)
            const int forced = eb ? atoi(eb) : 0;
            if (forced <= 0 && smem_for(p.tgy) <= budget) {
                const size_t sm1 = smem_for(p.tgy);
                FFB_CUDA(cudaFuncSetAttribute(prepare_onepass_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm1));
                prepare_onepass_kernel<false><<<p.Bp, PREP_CTA, sm1, as_stream(stream)>>>(q);
                FFB_CUDA(cudaGetLastError());
                return 0;
            }
            int rows = p.tgy;
            if (forced > 0) {
                rows = forced < p.tgy ? forced : p.tgy;
                while (smem_for(rows) > budget) --rows;
            } else {
                while (smem_for(rows) > budget) rows = (rows + 1) / 2;
            }
            q.band_rows = rows;
            const size_t smb = smem_for(rows);
            FFB_CUDA(cudaFuncSetAttribute(prepare_onepass_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smb));
            prepare_onepass_kernel<true><<<p.Bp, PREP_CTA, smb, as_stream(stream)>>>(q);
            FFB_CUDA(cudaGetLastError());
            return 0;
        }
        if (smem > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(prepare_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        prepare_kernel<true><<<p.Bp, PREP_CTA, smem, as_stream(stream)>>>(q);
    } else {
        if (smem > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(prepare_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        prepare_kernel<false><<<p.Bp, PREP_CTA, smem, as_stream(stream)>>>(q);
    }
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_splat_fwd(const ffb_splat_desc* d, const float* pts, const void* workspace,
                             float* out_sum, int sum_transposed, float* out_softor, void* stream) {
    (void)pts;
    Plan p;
    if (int rc = make_plan(d, &p)) return rc;
    if (!workspace) return fail_arg(FFB_E_ARG, "splat_fwd: null workspace");
    if (!out_sum && !out_softor) return fail_arg(FFB_E_ARG, "splat_fwd: no output requested");
    RasterParams q;
    fill_raster(d, p, workspace, q);
    q.out_sum = out_sum; q.out_softor = out_softor;
    cudaStream_t st = as_stream(stream);
    if (p.fast) {
        const WtConsts fc = wt_consts(d, p);
        const int B = d->B;
        const OvfParams ov = {q.ovf, q.ovf + 1, B};
        {
            // production path: finished tiles leave through TMA stores (needs 16-byte aligned bases and row pitches)
            const char* e = getenv("FFB_SPLAT_NO_TMA");
            CUtensorMap ms, mo;
            bool ok = !(e && e[0] == '1');
            const uint64_t t0 = (uint64_t)d->ts0, t1 = (uint64_t)d->ts1;
            if (ok && out_softor) ok = tma::encode_f32_3d(&mo, out_softor, t0, t1, (uint64_t)B, WT, WT, CU_TENSOR_MAP_SWIZZLE_NONE);
            if (ok && out_sum)
                ok = sum_transposed ? tma::encode_f32_3d(&ms, out_sum, t1, t0, (uint64_t)B, WT, WT, CU_TENSOR_MAP_SWIZZLE_64B)
                                    : tma::encode_f32_3d(&ms, out_sum, t0, t1, (uint64_t)B, WT, WT, CU_TENSOR_MAP_SWIZZLE_NONE);
            if (ok) {
                if (!out_softor) mo = ms;                   // unused maps still have to be valid kernel parameters
                if (!out_sum) ms = mo;
#define FFB_FT1(S, O, T, M) launch_fwd_tma(splat_fwd_tma<S, O, T, M>, splat_fwd_ovf<S, O, T, M>, q, fc, ov, B, st, ms, mo, sizeof(WarpStage<M ? 2 : 0>))
#define FFB_FT(S, O, T) (p.mask_o ? FFB_FT1(S, O, T, true) : FFB_FT1(S, O, T, false))
                if (out_sum && out_softor) return sum_transposed ? FFB_FT(true, true, true) : FFB_FT(true, true, false);
                if (out_sum) return sum_transposed ? FFB_FT1(true, false, true, false) : FFB_FT1(true, false, false, false);
                return FFB_FT(false, true, false);
#undef FFB_FT
#undef FFB_FT1
            }
        }
#define FFB_FWD1(S, O, T, M) launch_wt(splat_fwd_wt<S, O, T, M>, splat_fwd_ovf<S, O, T, M>, q, fc, ov, B, st)
#define FFB_FWD(S, O, T) (p.mask_o ? FFB_FWD1(S, O, T, true) : FFB_FWD1(S, O, T, false))
        if (out_sum && out_softor) return sum_transposed ? FFB_FWD(true, true, true) : FFB_FWD(true, true, false);
        if (out_sum) return sum_transposed ? FFB_FWD1(true, false, true, false) : FFB_FWD1(true, false, false, false);
        return FFB_FWD(false, true, false);
#undef FFB_FWD
#undef FFB_FWD1
    }
    if (out_sum && out_softor)
        return sum_transposed ? launch_raster(splat_fwd_kernel<true, true, true>, q, d->B, st)
                              : launch_raster(splat_fwd_kernel<true, true, false>, q, d->B, st);
    if (out_sum)
        return sum_transposed ? launch_raster(splat_fwd_kernel<true, false, true>, q, d->B, st)
                              : launch_raster(splat_fwd_kernel<true, false, false>, q, d->B, st);
    return launch_raster(splat_fwd_kernel<false, true, false>, q, d->B, st);
}

extern "C" int ffb_splat_bwd(const ffb_splat_desc* d, const float* pts, const void* workspace,
                             const float* g_sum, int sum_transposed, const float* g_softor, const float* saved_softor,
                             float* d_pts, void* stream) {
    (void)pts;
    Plan p;
    if (int rc = make_plan(d, &p)) return rc;
    if (!workspace || !d_pts) return fail_arg(FFB_E_ARG, "splat_bwd: null pointer");
    if (!g_sum && !g_softor) return fail_arg(FFB_E_ARG, "splat_bwd: no upstream gradient");
    RasterParams q;
    fill_raster(d, p, workspace, q);
    q.g_sum = g_sum; q.g_softor = g_softor; q.d_pts = d_pts;
    cudaStream_t st = as_stream(stream);
    FFB_CUDA(cudaMemsetAsync(d_pts, 0, (size_t)d->B * d->N * 2 * sizeof(float), st));
    const size_t gsm = (size_t)(CTA / 32) * KCACHE * WROWS * 32 * sizeof(float);
    if (p.fast) {
        const WtConsts fc = wt_consts(d, p);
        const int B = d->B;
        const OvfParams ov = {q.ovf, q.ovf + 1, B};
        const char* e = getenv("FFB_SPLAT_NO_TMA");         // tests: force the plain-load kernels
        const bool tma_ok = !(e && e[0] == '1');
        const uint64_t t0 = (uint64_t)d->ts0, t1 = (uint64_t)d->ts1;
        BwdMaps m;
        if (g_softor && p.mask_o) {
            // soft-OR window tighter than its no-op radius: upstream 16x16 tiles through TMA, the soft-OR product read back from the
            // forward's output when it is given, rebuilt otherwise
            q.saved_softor = saved_softor;
            bool ok = tma_ok && tma::encode_f32_3d(&m.go, g_softor, t0, t1, (uint64_t)B, WT, WT, CU_TENSOR_MAP_SWIZZLE_NONE);
            if (ok && saved_softor) ok = tma::encode_f32_3d(&m.sv, saved_softor, t0, t1, (uint64_t)B, WT, WT, CU_TENSOR_MAP_SWIZZLE_NONE);
            if (ok && g_sum)
                ok = sum_transposed ? tma::encode_f32_3d(&m.gs, g_sum, t1, t0, (uint64_t)B, WT, WT, CU_TENSOR_MAP_SWIZZLE_64B)
                                    : tma::encode_f32_3d(&m.gs, g_sum, t0, t1, (uint64_t)B, WT, WT, CU_TENSOR_MAP_SWIZZLE_NONE);
            if (ok) {
                if (!saved_softor) m.sv = m.go;             // unused maps still have to be valid kernel parameters
                if (!g_sum) m.gs = m.go;
#define FFB_TMA1(S, T, V) launch_bwd_tma(splat_bwd_tma<S, true, T, V>, splat_bwd_ovf<S, true, T, true, V>, q, fc, ov, B, st, m, \
                                         sizeof(WarpStage<2, true, false, 1>), sizeof(WarpStage<2, true, false, 1>) * WT_WARPS)
#define FFB_TMA(S, T) (saved_softor ? FFB_TMA1(S, T, true) : FFB_TMA1(S, T, false))
                if (g_sum) return sum_transposed ? FFB_TMA(true, true) : FFB_TMA(true, false);
                return FFB_TMA(false, false);
#undef FFB_TMA
#undef FFB_TMA1
            }
        } else {
            // production path: super-tile kernel, whole 64x16 blocks of the upstream arrays through TMA (needs 16-byte aligned bases and
            // row pitches).  The soft-OR product is rebuilt from the candidates (saved_softor is not read), as is the overflow kernel's.
            bool ok = tma_ok;
            if (ok && g_softor) ok = tma::encode_f32_3d(&m.go, g_softor, t0, t1, (uint64_t)B, 2 * WT, WT, CU_TENSOR_MAP_SWIZZLE_128B);
            if (ok && g_sum)
                ok = sum_transposed ? tma::encode_f32_3d(&m.gs, g_sum, t1, t0, (uint64_t)B, WT, 2 * WT, CU_TENSOR_MAP_SWIZZLE_64B)
                                    : tma::encode_f32_3d(&m.gs, g_sum, t0, t1, (uint64_t)B, 2 * WT, WT, CU_TENSOR_MAP_SWIZZLE_128B);
            if (ok) {
                if (!g_softor) m.go = m.gs;                 // unused maps still have to be valid kernel parameters
                if (!g_sum) m.gs = m.go;
                m.sv = m.ot = m.go;
                const size_t so = sizeof(WarpStage<1, true, false, 1>) * WT_WARPS;
                // the sum window's truncation is dropped where every truncated texel has g < 2^-22 (its share of d/dP is below 1e-6):
                // the gradient of the sum is then one addend of the same FFMA2 instead of two mask computations per visit
                const double edge = (double)p.H_s * (double)p.H_s / (double)d->sigma;
                const bool msk = g_sum && edge * edge < 15.25;
#define FFB_ST0(S, O, T, K)                                                                                                          \
    (q.eager ? launch_bwd_stp(splat_bwd_stp<S, O, T, K, ST_REBUILD>, splat_bwd_ovf<S, O, T, false, false>, q, fc, ov, B, st, m,       \
                              (size_t)StSmem<S, O, T, ST_REBUILD>::bytes, so, 8)                                                     \
             : launch_bwd_st(splat_bwd_st<S, O, T, K>, splat_bwd_ovf<S, O, T, false, false>, q, fc, ov, B, st, m,                    \
                             (size_t)StSmem<S, O, T, ST_REBUILD>::bytes, so))
#define FFB_ST(S, O, T) (msk ? FFB_ST0(S, O, T, true) : FFB_ST0(S, O, T, false))
                if (g_sum && g_softor) return sum_transposed ? FFB_ST(true, true, true) : FFB_ST(true, true, false);
                if (g_sum) return sum_transposed ? FFB_ST(true, false, true) : FFB_ST(true, false, false);
                return FFB_ST0(false, true, false, false);
#undef FFB_ST
#undef FFB_ST0
            }
        }
        // plain-load fallback: textures the TMA unit cannot describe (unaligned base, sides not multiples of 4)
        q.saved_softor = g_softor ? saved_softor : nullptr;
#define FFB_BWD1(S, O, T, M, V) launch_wt(splat_bwd_wt<S, O, T, M, V>, splat_bwd_ovf<S, O, T, M, V>, q, fc, ov, B, st, WB_CTA, \
                                          sizeof(WarpStage<M ? 2 : 1, true, true, 1>) * WB_WARPS, sizeof(WarpStage<M ? 2 : 1, true, false, 1>) * WT_WARPS)
#define FFB_BWD2(S, O, T, M) (q.saved_softor ? FFB_BWD1(S, O, T, M, true) : FFB_BWD1(S, O, T, M, false))
#define FFB_BWD(S, O, T) (p.mask_o ? FFB_BWD2(S, O, T, true) : FFB_BWD2(S, O, T, false))
        if (g_sum && g_softor) return sum_transposed ? FFB_BWD(true, true, true) : FFB_BWD(true, true, false);
        if (g_sum) return sum_transposed ? FFB_BWD1(true, false, true, false, false) : FFB_BWD1(true, false, false, false, false);
        return FFB_BWD(false, true, false);
#undef FFB_BWD
#undef FFB_BWD2
#undef FFB_BWD1
    }
    if (g_sum && g_softor)
        return sum_transposed ? launch_raster(splat_bwd_kernel<true, true, true>, q, d->B, st, gsm)
                              : launch_raster(splat_bwd_kernel<true, true, false>, q, d->B, st, gsm);
    if (g_sum)
        return sum_transposed ? launch_raster(splat_bwd_kernel<true, false, true>, q, d->B, st)
                              : launch_raster(splat_bwd_kernel<true, false, false>, q, d->B, st);
    return launch_raster(splat_bwd_kernel<false, true, false>, q, d->B, st, gsm);
}

extern "C" int ffb_splat_bwd_l1(const ffb_splat_desc* d, const float* pts, const void* workspace,
                                const float* out_sum, int sum_transposed, const float* out_softor,
                                float* loss_out, float* d_pts, void* stream) {
    (void)pts;
    Plan p;
    if (int rc = make_plan(d, &p)) return rc;
    if (!workspace || !d_pts || !out_sum || !out_softor || !loss_out) return fail_arg(FFB_E_ARG, "splat_bwd_l1: null pointer");
    if (sum_transposed && d->ts0 != d->ts1)
        return fail_arg(FFB_E_ARG, "splat_bwd_l1: softor [ts1,ts0] and a transposed sum [ts0,ts1] only pair elementwise on square textures");
    if (!p.fast || p.mask_o) return fail_arg(FFB_E_UNSUPPORTED, "splat_bwd_l1: needs the warp-tile path (texture larger than the footprints, exact soft-OR window)");
    RasterParams q;
    fill_raster(d, p, workspace, q);
    q.g_sum = out_sum; q.g_softor = out_softor; q.d_pts = d_pts;
    q.loss = loss_out; q.loss_inv = 1.0f / ((float)d->ts0 * (float)d->ts1);
    cudaStream_t st = as_stream(stream);
    const int B = d->B;
    // the super-tile kernel in its loss mode: whole 64x16 blocks of the forward's outputs, two request rounds per item when the sum is
    // stored transposed (mirrored index -> signs in shared memory, then own index)
    BwdMaps m;
    const uint64_t t0 = (uint64_t)d->ts0, t1 = (uint64_t)d->ts1;
    bool ok = tma::encode_f32_3d(&m.go, out_softor, t0, t1, (uint64_t)B, 2 * WT, WT, CU_TENSOR_MAP_SWIZZLE_128B);
    if (ok) ok = sum_transposed ? tma::encode_f32_3d(&m.gs, out_sum, t1, t0, (uint64_t)B, 2 * WT, WT, CU_TENSOR_MAP_SWIZZLE_128B)
                                : tma::encode_f32_3d(&m.gs, out_sum, t0, t1, (uint64_t)B, 2 * WT, WT, CU_TENSOR_MAP_SWIZZLE_128B);
    if (ok && sum_transposed)
        ok = tma::encode_f32_3d(&m.sv, out_sum, t1, t0, (uint64_t)B, WT, 2 * WT, CU_TENSOR_MAP_SWIZZLE_64B) &&
             tma::encode_f32_3d(&m.ot, out_softor, t0, t1, (uint64_t)B, WT, 2 * WT, CU_TENSOR_MAP_SWIZZLE_64B);
    else if (ok) { m.sv = m.gs; m.ot = m.go; }
    if (!ok) return fail_arg(FFB_E_UNSUPPORTED, "splat_bwd_l1: textures must be 16-byte aligned with sides that are multiples of 4 (TMA)");
    FFB_CUDA(cudaMemsetAsync(d_pts, 0, (size_t)B * d->N * 2 * sizeof(float), st));
    FFB_CUDA(cudaMemsetAsync(loss_out, 0, (size_t)B * sizeof(float), st));
    const WtConsts fc = wt_consts(d, p);
    const OvfParams ov = {q.ovf, q.ovf + 1, B};
    const size_t so = sizeof(WarpStage<1, true, false, 1>) * WT_WARPS;
    const double edge = (double)p.H_s * (double)p.H_s / (double)d->sigma;     // sum-window mask as in ffb_splat_bwd
    const bool msk = edge * edge < 15.25;
#define FFB_SL(T, K) launch_bwd_stp(splat_bwd_stp<true, true, T, K, ST_LOSS>, splat_bwd_ovf<true, true, T, false, true, true>, q, fc, ov, B, st, m, \
                                    (size_t)StSmem<true, true, T, ST_LOSS>::bytes, so, 0)
    if (sum_transposed) return msk ? FFB_SL(true, true) : FFB_SL(true, false);
    return msk ? FFB_SL(false, true) : FFB_SL(false, false);
#undef FFB_SL
}

extern "C" int ffb_reduce_over_samples(const float* in, int32_t B, int64_t row_elems, float* out, void* stream) {
    if (!in || !out || B <= 0 || row_elems <= 0) return fail_arg(FFB_E_ARG, "reduce_over_samples: bad argument");
    const unsigned grid = (unsigned)((row_elems + 31) / 32);
    reduce_samples_kernel<<<grid, 256, 0, as_stream(stream)>>>(in, B, row_elems, out);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_fold_allreduce(const float* in, int32_t B, int64_t row_elems, float* const* recv_bufs, uint32_t* const* flag_bufs,
                                  int32_t rank, int32_t world, uint32_t epoch, float* out, int32_t* err_flag, void* stream) {
    if (!in || !out || !recv_bufs || !flag_bufs || !err_flag || B <= 0 || row_elems <= 0) return fail_arg(FFB_E_ARG, "fold_allreduce: bad argument");
    if (world < 1 || world > 8 || rank < 0 || rank >= world) return fail_arg(FFB_E_LIMIT, "fold_allreduce: 1..8 ranks of one NVLink domain");
    if (epoch == 0) return fail_arg(FFB_E_ARG, "fold_allreduce: epochs start at 1 (the flag arrays start zeroed)");
    PeerTable pt;
    for (int r = 0; r < 8; ++r) {
        pt.recv[r] = r < world ? recv_bufs[r] : nullptr;
        pt.flag[r] = r < world ? flag_bufs[r] : nullptr;
        if (r < world && (!pt.recv[r] || !pt.flag[r])) return fail_arg(FFB_E_ARG, "fold_allreduce: null peer pointer");
    }
    const unsigned grid = (unsigned)((row_elems + 31) / 32);
    if (grid > (unsigned)kNumSMs * 8) return fail_arg(FFB_E_LIMIT, "fold_allreduce: every CTA of the launch must be resident (row_elems <= 37888)");
    fold_allreduce_kernel<<<grid, 256, 0, as_stream(stream)>>>(in, B, row_elems, pt, rank, world, epoch, out, err_flag);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_reduce_sample_groups(const float* in, int32_t B, int64_t row_elems, float* out, void* stream) {
    if (!in || !out || B <= 0 || row_elems <= 0) return fail_arg(FFB_E_ARG, "reduce_sample_groups: bad argument");
    if ((row_elems & 3) != 0 || ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15) != 0)
        return fail_arg(FFB_E_UNSUPPORTED, "reduce_sample_groups: rows must be 16-byte aligned multiples of 4 elements");
    const long long row4 = row_elems / 4;
    const int G = (B + 7) / 8;
    if (G > 65535) return fail_arg(FFB_E_LIMIT, "reduce_sample_groups: B > 524280");
    reduce_groups_kernel<<<dim3((unsigned)((row4 + 127) / 128), (unsigned)G), 256, 0, as_stream(stream)>>>(
        reinterpret_cast<const float4*>(in), B, row4, reinterpret_cast<float4*>(out));
    FFB_CUDA(cudaGetLastError());
    return 0;
}

static int dense_fwd_impl(const float* pts, int32_t N, int32_t ts0, int32_t ts1, float sx, float sy, float sigma, float* out, void* stream) {
    if (!pts || !out || N <= 0 || ts0 <= 0 || ts1 <= 0 || !(sigma > 0.f)) return fail_arg(FFB_E_ARG, "splat_dense_fwd: bad argument");
    const size_t total = (size_t)N * ts0 * ts1;
    size_t blocks = (total + 255) / 256;
    if (blocks > (size_t)kNumSMs * 32) blocks = (size_t)kNumSMs * 32;
    dense_fwd_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(pts, N, ts0, ts1, sx, sy, sigma, 1.0f / sigma, out);
    FFB_CUDA(cudaGetLastError());
    return 0;
}
static int dense_bwd_impl(const float* pts, int32_t N, int32_t ts0, int32_t ts1, float sx, float sy, float sigma, const float* g_out,
                          float* d_pts, void* stream) {
    if (!pts || !g_out || !d_pts || N <= 0 || ts0 <= 0 || ts1 <= 0 || !(sigma > 0.f)) return fail_arg(FFB_E_ARG, "splat_dense_bwd: bad argument");
    if (N > 65535) return fail_arg(FFB_E_LIMIT, "splat_dense_bwd: N > 65535");
    cudaStream_t st = as_stream(stream);
    FFB_CUDA(cudaMemsetAsync(d_pts, 0, (size_t)N * 2 * sizeof(float), st));
    const size_t frame = (size_t)ts0 * ts1;
    unsigned chunks = (unsigned)((frame + 256 * 16 - 1) / (256 * 16));
    if (chunks > 64) chunks = 64;
    if (chunks < 1) chunks = 1;
    dense_bwd_kernel<<<dim3(chunks, N), 256, 0, st>>>(pts, N, ts0, ts1, sx, sy, sigma, 1.0f / sigma, g_out, d_pts);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_splat_dense_fwd(const float* pts, int32_t N, int32_t ts0, int32_t ts1, float sigma, float* out, void* stream) {
    return dense_fwd_impl(pts, N, ts0, ts1, (float)ts0, (float)ts1, sigma, out, stream);
}
extern "C" int ffb_splat_dense_bwd(const float* pts, int32_t N, int32_t ts0, int32_t ts1, float sigma,
                                   const float* g_out, float* d_pts, void* stream) {
    return dense_bwd_impl(pts, N, ts0, ts1, (float)ts0, (float)ts1, sigma, g_out, d_pts, stream);
}
extern "C" int ffb_splat_dense_px_fwd(const float* pts, int32_t N, int32_t ts0, int32_t ts1, float sigma, float* out, void* stream) {
    return dense_fwd_impl(pts, N, ts0, ts1, 1.f, 1.f, sigma, out, stream);
}
extern "C" int ffb_splat_dense_px_bwd(const float* pts, int32_t N, int32_t ts0, int32_t ts1, float sigma,
                                      const float* g_out, float* d_pts, void* stream) {
    return dense_bwd_impl(pts, N, ts0, ts1, 1.f, 1.f, sigma, g_out, d_pts, stream);
}

extern "C" int ffb_l1_loss_fwd_bwd(const float* a, const float* b, int b_transposed, int32_t B, int32_t ts0, int32_t ts1,
                                   float* loss_out, float* g_a, float* g_b, void* stream) {
    if (!a || !b || !loss_out || B <= 0 || ts0 <= 0 || ts1 <= 0) return fail_arg(FFB_E_ARG, "l1_loss: bad argument");
    if (B > 65535) return fail_arg(FFB_E_LIMIT, "l1_loss: B > 65535");
    cudaStream_t st = as_stream(stream);
    FFB_CUDA(cudaMemsetAsync(loss_out, 0, (size_t)B * sizeof(float), st));
    const unsigned tiles = (unsigned)(((ts0 + 31) / 32) * ((ts1 + 31) / 32));
    const float inv = 1.0f / ((float)ts0 * (float)ts1);
    if (b_transposed) l1_kernel<true><<<dim3(tiles, B), 256, 0, st>>>(a, b, ts0, ts1, inv, loss_out, g_a, g_b);
    else l1_kernel<false><<<dim3(tiles, B), 256, 0, st>>>(a, b, ts0, ts1, inv, loss_out, g_a, g_b);
    FFB_CUDA(cudaGetLastError());
    return 0;
}
