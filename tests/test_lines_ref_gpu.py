"""The line and depth rasterisers (fireflies_b200/csrc/ffb_lines.cu) against a plain fp64 restatement of the reference
arithmetic, evaluated on the CPU with torch autograd, at the shapes where the kernels' tiling, line staging and culling
have edges: line counts across the 128-line staging chunk and its 64-line halves, textures that are not multiples of
the 32-column x 64-row CTA tile, culling radii from nearly nothing to most of the frame, degenerate and exactly placed
segments, every sum / soft-OR kernel instantiation, unaligned storage, and the depth rasteriser's clamped maximum and
256-point staging loop.

Tolerances: forward 1e-5 relative + 1e-6 absolute; gradients 1e-4 relative + 1e-4 of the largest reference component.
The line forwards also allow, per texel, the distance between the reference's own float32 arithmetic (the CPU oracle,
which the kernels restate op for op) and fp64: its x - (a + t0 m) cancels at the scale of the frame, so at sigma 0.5 on
a 257-wide frame float32 alone is 1.2e-4 relative from fp64 (4e-5 at 100 wide, below 1e-5 from sigma 10 on).
Every gradient check also requires a nonzero kernel gradient for each line / point whose reference gradient is nonzero
(norm above 1e-12 of the largest; below that sit the tails past the kernels' exp(-87) cut-off), so a dropped gradient
write fails whatever its size."""
import math

import pytest
import torch

from oracle import ff_oracle as O

pytestmark = pytest.mark.gpu

F64 = torch.float64
EPS32 = float(torch.finfo(torch.float32).eps)       # the reference's torch.finfo().eps (default dtype float32)
TILE = (32, 64)                                     # CTA tile of the fused line kernels: columns, rows


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import fireflies_b200.graphics.rasterization as R
    return R


# ---- fp64 reference (oracle/ff_oracle.py's arithmetic without its float32 casts) ------------------------------------
def ref_lines(lines, sigma, ts):
    """rasterize_lines (reference rasterization.py:107-153): ``[L, ts1, ts0]``, exp(-(d2*d2)/(sigma*sigma))."""
    ts0, ts1 = ts
    scale = torch.tensor([ts0, ts1], dtype=F64)
    a = (lines[:, 0, :] * scale).T[:, :, None, None]                  # [2, L, 1, 1]
    b = (lines[:, 1, :] * scale).T[:, :, None, None]
    y, x = torch.meshgrid(torch.arange(ts1, dtype=F64), torch.arange(ts0, dtype=F64), indexing="ij")
    xy = torch.stack([x, y])[:, None]                                  # [2, 1, ts1, ts0]
    pa, pb, m = xy - a, xy - b, b - a
    t0 = (pa * m).sum(0) / ((m * m).sum(0) + EPS32)
    patm = xy - (a + t0[None] * m)
    d = (t0 <= 0) * (pa * pa).sum(0) + (t0 > 0) * (t0 < 1) * (patm * patm).sum(0) + (t0 >= 1) * (pb * pb).sum(0)
    return torch.exp(-(d * d) / (sigma * sigma))


def ref_depth(points, depth, sigma, ts):
    """rasterize_depth (reference rasterization.py:66-104): the splat normalised by its maximum over the frame, times depth."""
    ts0, ts1 = ts
    P = points * torch.tensor([ts0, ts1], dtype=F64)
    dc = torch.arange(ts0, dtype=F64).view(1, 1, ts0) - P[:, 0].view(-1, 1, 1)
    dr = torch.arange(ts1, dtype=F64).view(1, ts1, 1) - P[:, 1].view(-1, 1, 1)
    u = (dc * dc + dr * dr) / sigma
    g = torch.exp(-(u * u))
    g = g / g.max(dim=2, keepdim=True)[0].max(dim=1, keepdim=True)[0]
    return g * depth.reshape(-1, 1, 1)


def ref_softor(tex):
    return 1 - torch.prod(1 - tex, dim=0)


# ---- checks ---------------------------------------------------------------------------------------------------------
def ranges(idx):
    """[64, 65, ..., 127, 192, ...] -> '64..127, 192..199'"""
    idx, out, i = [int(v) for v in idx], [], 0
    while i < len(idx):
        j = i
        while j + 1 < len(idx) and idx[j + 1] == idx[j] + 1:
            j += 1
        out.append(f"{idx[i]}..{idx[j]}" if j > i else f"{idx[i]}")
        i = j + 1
    return ", ".join(out)


def fwd_close(got, want, rtol=1e-5, atol=1e-6, f32=None):
    """``f32``: the same quantity in the reference's float32 arithmetic; its distance from ``want`` is allowed on top."""
    got, want = got.detach().cpu().double(), want.detach().cpu().double()
    assert got.shape == want.shape, (got.shape, want.shape)
    if f32 is not None:
        atol = atol + (f32.detach().double() - want).abs()
    err = (got - want).abs() - (atol + rtol * want.abs())
    worst = int(err.argmax()) if err.numel() else 0
    assert not (err.max() > 0) and not err.isnan().any(), \
        f"max violation {float(err.max()):.3e} at flat index {worst}: got {float(got.flatten()[worst]):.9g}, " \
        f"want {float(want.flatten()[worst]):.9g}"


def grad_close(got, want, what="line"):
    got = got.detach().cpu().double().reshape(got.shape[0], -1)
    want = want.detach().cpu().double().reshape(want.shape[0], -1)
    assert got.shape == want.shape, (got.shape, want.shape)
    norm = want.norm(dim=1)
    lost = (norm > 1e-12 * norm.max()) & (norm > 0) & (got == 0).all(dim=1)
    assert not lost.any(), f"{what}s with a nonzero reference gradient but an all-zero kernel gradient " \
                           f"({int(lost.sum())} of {got.shape[0]}): {ranges(lost.nonzero().flatten())}"
    atol = 1e-4 * float(want.abs().max())
    err = (got - want).abs() - (atol + 1e-4 * want.abs())
    worst = int(err.argmax())
    assert not (err.max() > 0) and not err.isnan().any(), \
        f"max violation {float(err.max()):.3e} at {what} {worst // got.shape[1]}: got {got.flatten()[worst].item():.9g}, " \
        f"want {want.flatten()[worst].item():.9g} (largest reference component {atol * 1e4:.3e})"


# ---- inputs ---------------------------------------------------------------------------------------------------------
def grid(t):
    """Round frame-relative coordinates to multiples of 2^-12: then ``coordinate * texture_size`` is exact in float32 for
    texture sides below 2^11, and the comparison measures the kernels' arithmetic rather than the rounding of the
    scaled input (which alone moves a texel value by up to 2e-5 relative against fp64)."""
    return (t.double() * 4096).round().float() / 4096


def rand_lines(L, seed, lo=-0.1, hi=1.1):
    """Half long segments across the frame, half short ones (a tenth of the frame), end points in [lo, hi]."""
    gen = torch.Generator().manual_seed(seed)
    a = torch.rand(L, 2, generator=gen) * (hi - lo) + lo
    b = torch.rand(L, 2, generator=gen) * (hi - lo) + lo
    short = torch.arange(L) % 2 == 1
    b[short] = a[short] + (torch.rand(int(short.sum()), 2, generator=gen) - 0.5) * 0.2
    return grid(torch.stack([a, b], dim=1))


def texel_lines(segs, ts):
    """Segments given in texel units, normalised so that the kernels' ``lines * texture_size`` recovers them exactly."""
    t = torch.tensor(segs, dtype=torch.float64)
    n = (t / torch.tensor([ts[0], ts[1]], dtype=torch.float64)).float()
    assert torch.equal(n.double() * torch.tensor([ts[0], ts[1]], dtype=torch.float64), t), "not exactly representable"
    return n


def weights(ts, seed, n=2):
    gen = torch.Generator().manual_seed(seed)
    return [torch.randn(ts[1], ts[0], generator=gen) for _ in range(n)]


def run_reduce(R, lines, sigma, ts, wS, wO):
    """lines_reduce with the named reductions (None = not requested): forward outputs and d(sum wS*s + wO*o)/d lines,
    for the kernel and for the fp64 reference."""
    reduce = tuple(n for n, w in (("sum", wS), ("softor", wO)) if w is not None)
    l = lines.cuda().requires_grad_(True)
    s, o = R.lines_reduce(l, sigma, ts, reduce=reduce)
    loss = sum((x * w.cuda()).sum() for x, w in ((s, wS), (o, wO)) if w is not None)
    loss.backward()
    l64 = lines.double().requires_grad_(True)
    tex = ref_lines(l64, sigma, ts)
    S, So = tex.sum(0), ref_softor(tex)
    sum((x * w.double()).sum() for x, w in ((S, wS), (So, wO)) if w is not None).backward()
    return (s, o, l.grad), (S, So, l64.grad)


def check_lines_fwd(s, o, S, So, lines, sigma, ts):
    t32 = O.rasterize_lines(lines, sigma, ts)
    if s is not None:
        fwd_close(s, S, f32=t32.sum(0))
    if o is not None:
        fwd_close(o, So, f32=O.softor(t32))


def check_reduce(R, lines, sigma, ts, seed=0):
    wS, wO = weights(ts, seed)
    (s, o, g), (S, So, G) = run_reduce(R, lines, sigma, ts, wS, wO)
    check_lines_fwd(s, o, S, So, lines, sigma, ts)
    grad_close(g, G)


# ---- fused sum / soft-OR ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", [1, 63, 64, 65, 127, 128, 129, 200, 300])
def test_reduce_line_counts(R, L):
    """Across the 128-line staging chunk: the backward flushes 4 gradient components per staged line with 256 threads."""
    check_reduce(R, rand_lines(L, seed=L), 6.0, [100, 70], seed=L)


@pytest.mark.parametrize("reduce", [("sum",), ("softor",), ("sum", "softor")])
def test_reduce_instantiations(R, reduce):
    """Each sum / soft-OR kernel instantiation against fp64, and against the both-outputs kernels."""
    ts, sigma, L = [100, 70], 4.0, 200
    lines = rand_lines(L, seed=5)
    wS, wO = weights(ts, seed=5)
    wS, wO = (wS if "sum" in reduce else None), (wO if "softor" in reduce else None)
    (s, o, g), (S, So, G) = run_reduce(R, lines, sigma, ts, wS, wO)
    check_lines_fwd(s, o, S, So, lines, sigma, ts)
    grad_close(g, G)
    s2, o2 = R.lines_reduce(lines.cuda(), sigma, ts)
    for got, both in ((s, s2), (o, o2)):
        assert got is None or torch.equal(got, both), "single-output forward differs from the both-outputs forward"
    if len(reduce) == 1:
        # one upstream gradient == both upstream gradients with the other one zero
        l = lines.cuda().requires_grad_(True)
        s2, o2 = R.lines_reduce(l, sigma, ts)
        zero = torch.zeros(ts[1], ts[0])
        ((s2 * (wS if wS is not None else zero).cuda()).sum() + (o2 * (wO if wO is not None else zero).cuda()).sum()).backward()
        assert float((g - l.grad).norm()) <= 1e-6 * float(l.grad.norm()), float((g - l.grad).norm() / l.grad.norm())


@pytest.mark.parametrize("ts", [[1, 1], [31, 7], [33, 65], [257, 129]], ids=lambda t: f"{t[0]}x{t[1]}")
def test_reduce_ragged_textures(R, ts):
    """Textures smaller than, or ragged against, the 32 x 64 tile.  The native calls run on buffers followed by
    sentinels: the forward must write only the frame, the backward must read only the frame (NaN past it)."""
    from fireflies_b200 import _native as nat
    L, sigma = 70, 2.0
    lines = rand_lines(L, seed=ts[0])
    wS, wO = weights(ts, seed=ts[1])
    (s, o, g), (S, So, G) = run_reduce(R, lines, sigma, ts, wS, wO)
    check_lines_fwd(s, o, S, So, lines, sigma, ts)
    grad_close(g, G)
    n, pad = ts[0] * ts[1], TILE[1] * ts[0] + TILE[0]
    ln = lines.cuda()
    out = torch.full((2, n + pad), 12345.0, device="cuda")
    nat.check(nat.lib().ffb_lines_reduce_fwd(ln.data_ptr(), L, ts[0], ts[1], sigma, out[0].data_ptr(), out[1].data_ptr(),
                                             nat.stream()), "ffb_lines_reduce_fwd")
    assert (out[:, n:] == 12345.0).all(), "the forward wrote past the frame"
    assert torch.equal(out[0, :n].view(ts[1], ts[0]), s) and torch.equal(out[1, :n].view(ts[1], ts[0]), o)
    gin = torch.full((2, n + pad), float("nan"), device="cuda")
    gin[0, :n], gin[1, :n] = wS.cuda().flatten(), wO.cuda().flatten()
    d = torch.empty(L, 2, 2, device="cuda")
    nat.check(nat.lib().ffb_lines_reduce_bwd(ln.data_ptr(), L, ts[0], ts[1], sigma, gin[0].data_ptr(), gin[1].data_ptr(),
                                             d.data_ptr(), nat.stream()), "ffb_lines_reduce_bwd")
    grad_close(d, G)


@pytest.mark.parametrize("sigma", [0.5, 2.0, 10.0, 400.0])
def test_reduce_culling_radius(R, sigma):
    """sigma 0.5 culls nearly every (warp block, line) pair, 400 almost none (exp(-d2^2/sigma^2) spans most of the frame)."""
    check_reduce(R, rand_lines(100, seed=int(sigma * 10)), sigma, [100, 70], seed=3)


@pytest.mark.parametrize("sigma", [0.5, 2.0, 10.0, 400.0])
def test_reduce_culling_block_corner(R, sigma):
    """A segment off the frame's top-left corner, on the far side of texel (0, 0) from the centre of the 8 x 32 warp block
    that holds it, at the distance where exp(-d2^2/sigma^2) = exp(-50): just inside the culling radius `cut` of that texel,
    while the block's centre is 16 texels farther.  The culling test must keep the pair: the segment's only gradient comes
    from there (about 1e-20, seen by the nonzero check, not by the tolerance)."""
    ts = [100, 70]
    c = torch.tensor([15.5, 3.5], dtype=F64)                # centre of the warp block with rows 0..7, columns 0..31
    u = c / c.norm()
    D = 50 ** 0.25 * math.sqrt(sigma)                        # distance of the segment from texel (0, 0)
    assert D < math.sqrt(sigma * math.sqrt(88.0) * 1.01)     # inside the kernels' cut
    p, perp = -D * u, torch.stack([-u[1], u[0]])
    seg = torch.stack([p - 0.5 * perp, p + 0.5 * perp]) / torch.tensor(ts, dtype=F64)
    lines = grid(seg)[None]
    far = rand_lines(3, seed=1, lo=0.6, hi=0.9)              # far from the corner, inside the frame
    for ls in (lines, torch.cat([far, lines])):
        wS, wO = weights(ts, seed=int(sigma))
        (s, o, g), (S, So, G) = run_reduce(R, ls, sigma, ts, wS, wO)
        assert float(G[-1].norm()) > 0
        check_lines_fwd(s, o, S, So, ls, sigma, ts)
        grad_close(g[-1:], G[-1:])
        grad_close(g, G)


# ---- geometry edges ----------------------------------------------------------------------------------------------------
EDGE_TS = [72, 40]          # texel x = 9k and y = 5k are exact as k/8 of the frame


def edge_lines():
    segs = [
        [[18, 10], [18, 10]],          # degenerate on a texel centre (the eps guard; d2 = 0 there)
        [[9, 5], [36, 5]],             # end points on texel centres: t0 exactly 0 and 1 at their texels
        [[9, 10], [36, 25]],           # the same, diagonal (m.m = 954 exactly)
        [[36, 20], [54, 20]],          # three lines through texel (45, 20): z2 with three zero factors
        [[45, 10], [45, 30]],
        [[36, 15], [54, 25]],
    ]
    lines = texel_lines(segs, EDGE_TS)
    more = grid(torch.tensor([
        [[0.3137, 0.6211], [0.3137, 0.6211]],     # degenerate, off the texel grid
        [[-0.5, -0.3], [-0.2, -0.6]],              # entirely outside the frame, far
        [[1.02, 0.2], [1.09, 0.8]],                # entirely outside the frame, within reach of the last columns
        [[0.4, -0.07], [0.7, -0.02]],              # outside, above the first row
        [[-0.3, 0.5], [1.4, 0.6]],                 # end points outside [0, 1], crossing the frame
        [[0.2, 1.3], [0.9, -0.25]],
    ]))
    return torch.cat([lines, more])


@pytest.mark.parametrize("sigma", [1.0, 6.0])
def test_reduce_geometry_edges(R, sigma):
    check_reduce(R, edge_lines(), sigma, EDGE_TS, seed=11)


@pytest.mark.parametrize("sigma", [1.0, 6.0])
def test_dense_geometry_edges(R, sigma):
    lines = edge_lines()
    l = lines.cuda().requires_grad_(True)
    tex = R.rasterize_lines(l, sigma, EDGE_TS)
    w = torch.randn(tex.shape, generator=torch.Generator().manual_seed(2))
    (tex * w.cuda()).sum().backward()
    l64 = lines.double().requires_grad_(True)
    ref = ref_lines(l64, sigma, EDGE_TS)
    (ref * w.double()).sum().backward()
    fwd_close(tex, ref, f32=O.rasterize_lines(lines, sigma, EDGE_TS))
    grad_close(l.grad, l64.grad)


def test_softor_two_exact_zeros_and_a_rounded_one(R):
    """Two segments exactly through texel (20, 20) and a third 2^-10 texels from it, where 1 - g rounds to 0 in float32
    but its distance term does not vanish.  torch.prod's backward gives every factor at that texel a zero soft-OR
    gradient (at least two other factors are 0), so with the upstream gradients a unit impulse there, the third segment's
    gradient is its sum term alone, and the first two get (next to) nothing."""
    ts, sigma = [64, 32], 1.0
    d = 2.0 ** -10
    lines = texel_lines([[[10, 20], [30, 20]], [[20, 10], [20, 30]], [[10, 20 + d], [30, 20 + d]]], ts)
    w = torch.zeros(ts[1], ts[0])
    w[20, 20] = 1.0
    (s, o, g), (S, So, G) = run_reduce(R, lines, sigma, ts, w, w)
    check_lines_fwd(s, o, S, So, lines, sigma, ts)
    assert float(G[2].norm()) > 1e3 * float(G[:2].norm())
    grad_close(g, G)


# ---- dense API and its relation to the fused reductions ----------------------------------------------------------------
def test_dense_lines_many(R):
    ts, sigma, L = [48, 36], 3.0, 300
    lines = rand_lines(L, seed=21)
    l = lines.cuda().requires_grad_(True)
    tex = R.rasterize_lines(l, sigma, ts)
    w = torch.randn(tex.shape, generator=torch.Generator().manual_seed(22))
    (tex * w.cuda()).sum().backward()
    l64 = lines.double().requires_grad_(True)
    ref = ref_lines(l64, sigma, ts)
    (ref * w.double()).sum().backward()
    fwd_close(tex, ref, f32=O.rasterize_lines(lines, sigma, ts))
    grad_close(l.grad, l64.grad)
    s, o = R.lines_reduce(lines.cuda(), sigma, ts)
    fwd_close(s, tex.detach().sum(0))
    fwd_close(o, R.softor(tex.detach()))


def test_lines_unaligned_storage(R):
    """A contiguous [L, 2, 2] view one float into its buffer: the kernels read lines as float4, the wrapper re-homes it."""
    ts, sigma, L = [100, 70], 4.0, 70
    lines = rand_lines(L, seed=31)
    buf = torch.empty(4 * L + 1, device="cuda")
    buf[1:] = lines.cuda().flatten()
    lu = buf[1:].view(L, 2, 2)
    assert lu.data_ptr() % 16 != 0
    s, o = R.lines_reduce(lu, sigma, ts)
    s2, o2 = R.lines_reduce(lines.cuda(), sigma, ts)
    assert torch.equal(s, s2) and torch.equal(o, o2)
    assert torch.equal(R.rasterize_lines(lu, sigma, ts), R.rasterize_lines(lines.cuda(), sigma, ts))
    leaf = buf[1:].view(L, 2, 2).detach().requires_grad_(True)
    wS, wO = weights(ts, seed=31)
    s, o = R.lines_reduce(leaf, sigma, ts)
    ((s * wS.cuda()).sum() + (o * wO.cuda()).sum()).backward()
    _, (_, _, G) = run_reduce(R, lines, sigma, ts, wS, wO)
    grad_close(leaf.grad, G)


# ---- depth ----------------------------------------------------------------------------------------------------------
def depth_points(N, sigma, ts, seed):
    """Texture-unit points: outside each side and corner (nearest in-frame texel clamped), a few texel centres plus a
    small offset, the rest random over and around the frame.  Fractional parts stay at least 0.05 from 0.5: at an exact
    midpoint torch's max backward and the kernel's rintf pick different (equally near) texels, both legitimately."""
    ts0, ts1 = ts
    D = 0.6 * math.sqrt(sigma)                 # off the frame by this much: the nearest texel keeps exp(-0.13)
    special = [[-D, 0.37 * ts1], [ts0 - 1 + D, 0.61 * ts1], [0.43 * ts0, -D], [0.29 * ts0, ts1 - 1 + D],
               [-0.8 * D, -0.6 * D], [ts0 - 1 + 0.7 * D, -0.6 * D], [-0.6 * D, ts1 - 1 + 0.8 * D],
               [ts0 - 1 + 0.75 * D, ts1 - 1 + 0.65 * D],
               [7.01, 5.0 - 0.02], [11 - 0.003, 3 + 0.004], [ts0 // 2 + 0.02, ts1 // 2]]
    gen = torch.Generator().manual_seed(seed)
    rnd = torch.rand(max(N - len(special), 0), 2, generator=gen, dtype=F64) * torch.tensor([ts0 + 2.0, ts1 + 2.0], dtype=F64) - 1
    P = torch.cat([torch.tensor(special, dtype=F64), rnd])[:N]
    frac = P - P.floor()
    P = torch.where((frac - 0.5).abs() < 0.05, P + 0.1, P)
    return (P / torch.tensor([ts0, ts1], dtype=F64)).float()


@pytest.mark.parametrize("N", [1, 65, 300])
@pytest.mark.parametrize("sigma", [1.0, 6.0, 200.0])
def test_depth_dense(R, N, sigma):
    ts = [37, 29]
    pts = depth_points(N, sigma, ts, seed=N)
    gen = torch.Generator().manual_seed(N + 1)
    dv = torch.rand(N, 1, generator=gen) + 0.2
    w = torch.randn(N, ts[1], ts[0], generator=gen)
    pc, dc = pts.cuda().requires_grad_(True), dv.cuda().requires_grad_(True)
    out = R.rasterize_depth(pc, dc, sigma, ts)
    (out * w.cuda()).sum().backward()
    p64, d64 = pts.double().requires_grad_(True), dv.double().requires_grad_(True)
    ref = ref_depth(p64, d64, sigma, ts)
    (ref * w.double()).sum().backward()
    fwd_close(out, ref)
    grad_close(pc.grad, p64.grad, what="point")
    grad_close(dc.grad, d64.grad, what="point")


@pytest.mark.parametrize("N", [255, 256, 257, 600])
def test_subsampled_point_raster(R, N):
    """Across the 256-point staging loop, odd sensor sides (81 -> 40 -> 20, 47 -> 23 -> 11), depths above 1."""
    sensor, sigma, levels = [81, 47], 6.0, 3
    pts = depth_points(N, sigma, sensor, seed=N)
    dv = torch.rand(N, 1, generator=torch.Generator().manual_seed(N)) * 1.6 + 0.2
    got = R.subsampled_point_raster(torch.cat([pts, dv], 1).cuda(), levels, sigma, sensor)
    assert len(got) == levels
    for i, lv in enumerate(got):
        ts = [sensor[0] // 2 ** i, sensor[1] // 2 ** i]
        want = 1 - torch.prod(1 - ref_depth(pts.double(), dv.double(), sigma, ts), dim=0, keepdim=True)
        fwd_close(lv, want)
