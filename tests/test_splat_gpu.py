"""GPU parity: the CUDA splat (through the C ABI) vs the CPU oracle and the reference-generated fixtures.

Tolerances (north star): forward 1e-5 relative, gradients 1e-4 relative, integer outputs bit-exact.
Forward comparisons add an absolute floor of 1e-6 (values are O(1); the reference's own dense and baked
variants differ from each other by 2.4e-7, SURVEY.md KAT5).  Gradient comparisons (`close_grad`) are per component:
|d - ref| <= 1e-4 |ref| + 1e-4 ||ref_n||, ref_n the gradient of the SAME point -- a point's two components are sums of the same
~1400 signed texel terms, so a component that cancels to near zero is judged against its point's gradient, never against the
largest gradient of the pattern.
"""
import numpy as np
import pytest
import torch

from oracle import ff_oracle as O

pytestmark = pytest.mark.gpu

SPLAT_CASES = ["splat_kat1", "splat_small_rect", "splat_mid", "splat_c1"]


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import fireflies_b200.graphics.rasterization as R
    return R


def T(a):
    return torch.from_numpy(np.asarray(a))


def close(a, b, rtol=1e-5, atol=1e-6):
    a = a.detach().cpu().double().numpy() if torch.is_tensor(a) else np.asarray(a, np.float64)
    b = b.detach().cpu().double().numpy() if torch.is_tensor(b) else np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    err = np.abs(a - b) - (atol + rtol * np.abs(b))
    assert err.max() <= 0, f"max violation {err.max():.3e}; max abs diff {np.abs(a - b).max():.3e}"


def close_grad(got, ref, rtol=1e-4):
    """per component: |got - ref| <= rtol |ref| + rtol max(||ref[point]||_2, 0.1 mean_m ||ref[m]||_2).  The second term's floor is for
    points whose gradient cancels (a component is a sum of ~1400 signed texel terms; the L1 gradients are sums of +-1/numel terms):
    such a point is judged against a tenth of the pattern's MEAN gradient norm -- never against the largest gradient."""
    a = got.detach().cpu().double().numpy() if torch.is_tensor(got) else np.asarray(got, np.float64)
    b = ref.detach().cpu().double().numpy() if torch.is_tensor(ref) else np.asarray(ref, np.float64)
    assert a.shape == b.shape and a.shape[-1] == 2, (a.shape, b.shape)
    nrm = np.linalg.norm(b, axis=-1, keepdims=True)
    scale = np.maximum(nrm, 0.1 * nrm.mean())
    err = np.abs(a - b) - (rtol * np.abs(b) + rtol * scale)
    worst = np.unravel_index(np.argmax(err), err.shape)
    assert err.max() <= 0, (f"max violation {err.max():.3e} at {worst}: got {a[worst]:.6e}, ref {b[worst]:.6e}, point norm "
                            f"{nrm[worst[:-1]][0]:.3e}, mean norm {nrm.mean():.3e}")


@pytest.mark.parametrize("case", SPLAT_CASES)
def test_forward_vs_reference_fixtures(R, golden, case):
    g = golden(case)
    pts, sigma, ts, st = T(g["points"]).cuda(), float(g["sigma"]), g["texture_size"].tolist(), int(g["stride"])
    close(R.baked_sum(pts, sigma, ts)[::st, ::st], g["baked_sum"])
    close(R.baked_sum_2(pts, sigma, ts)[::st, ::st], g["baked_sum_2"])
    close(R.baked_softor(pts, sigma, ts)[::st, ::st], g["baked_softor"])
    close(R.baked_softor_2(pts, sigma, ts)[::st, ::st], g["baked_softor_2"])
    if "dense_sum" in g:
        close(R.rasterize_points_baked_sum(pts, sigma, ts)[::st, ::st], g["dense_sum"])
        close(R.rasterize_points_baked_softor(pts, sigma, ts)[::st, ::st], g["dense_softor"])
    if "dense" in g:
        close(R.rasterize_points(pts, sigma, T(np.array(ts))), g["dense"], atol=1e-7)
    # fused: both reductions from one launch equal the separate calls bit for bit
    s, o = R.splat_reduce(pts, sigma, ts, sum_transposed=True)
    assert torch.equal(s, R.baked_sum_2(pts, sigma, ts)) and torch.equal(o, R.baked_softor_2(pts, sigma, ts))


@pytest.mark.parametrize("case", SPLAT_CASES)
def test_backward_vs_reference_fixtures(R, golden, case):
    g = golden(case)
    pts, sigma, ts = T(g["points"]).cuda(), float(g["sigma"]), g["texture_size"].tolist()
    h, w = ts[1], ts[0]
    if "wS" in g:
        wS, wO = T(g["wS"]), T(g["wO"])
    else:
        gen = torch.Generator().manual_seed(7)
        wS, wO = torch.randn(h, w, generator=gen), torch.randn(h, w, generator=gen)
    wS, wO = wS.cuda(), wO.cuda()
    # <wS, baked_sum> + <wO, baked_softor>
    p = pts.clone().requires_grad_(True)
    s, o = R.splat_reduce(p, sigma, ts)
    ((s * wS).sum() + (o * wO).sum()).backward()
    ref = g["baked_weighted_grad"]
    close_grad(p.grad, ref)
    # same through the transposed-sum layout (baked_sum_2): upstream gradient arrives transposed
    p = pts.clone().requires_grad_(True)
    s, o = R.splat_reduce(p, sigma, ts, sum_transposed=True)
    ((s * wS.T).sum() + (o * wO).sum()).backward()
    close_grad(p.grad, ref)
    # dense semantics
    if "dense_weighted_grad" in g:
        p = pts.clone().requires_grad_(True)
        s, o = R.splat_reduce(p, sigma, ts, num_std_sum=None, num_std_softor=None)
        ((s * wS).sum() + (o * wO).sum()).backward()
        ref = g["dense_weighted_grad"]
        close_grad(p.grad, ref)
    # the in-tree pattern-optimisation step: L1(baked_softor_2, baked_sum_2)
    if ts[0] == ts[1]:
        p = pts.clone().requires_grad_(True)
        s, o = R.splat_reduce(p, sigma, ts, sum_transposed=True, batch=1)
        loss = R.l1_loss(o, s, b_transposed=False)      # the reference compares softor with the *transposed* sum as-is
        loss.sum().backward()
        close(loss[0], g["baked_l1"], rtol=1e-5, atol=1e-8)
        ref = g["baked_l1_grad"]
        close_grad(p.grad, ref)


def test_dense_autograd_kat1(R, golden):
    g = golden("splat_kat1")
    pts, ts = T(g["points"]).cuda().requires_grad_(True), g["texture_size"].tolist()
    d = R.rasterize_points(pts, 4.0, T(np.array(ts)))
    loss = torch.nn.L1Loss()(R.softor(d), R.sum(d))
    loss.backward()
    close(loss, g["dense_l1"], rtol=1e-5, atol=1e-8)
    close(pts.grad, g["dense_l1_grad"], rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("n,ts,sigma,seed", [
    (1, [7, 5], 2.0, 0), (33, [100, 37], 12.5, 1), (300, [257, 129], 40.0, 2), (64, [64, 64], 225.0, 3), (500, [512, 512], 100.0, 4),
])
def test_randomised_vs_oracle(R, n, ts, sigma, seed):
    gen = torch.Generator().manual_seed(seed)
    pts = torch.rand(n, 2, generator=gen)
    wS, wO = torch.randn(ts[1], ts[0], generator=gen), torch.randn(ts[1], ts[0], generator=gen)
    p = pts.cuda().requires_grad_(True)
    s, o = R.splat_reduce(p, sigma, ts)
    close(s, O.baked_sum(pts, sigma, ts))
    close(o, O.baked_softor(pts, sigma, ts))
    ((s * wS.cuda()).sum() + (o * wO.cuda()).sum()).backward()
    pr = pts.clone().requires_grad_(True)
    ((O.baked_sum(pr, sigma, ts) * wS).sum() + (O.baked_softor(pr, sigma, ts) * wO).sum()).backward()
    close_grad(p.grad, pr.grad)
    # integer outputs: clip windows bit-exact
    win = R.splat_windows(pts.cuda(), sigma, ts).cpu()
    assert torch.equal(win[:, 0], O.baked_windows(pts, sigma, ts, 4))
    assert torch.equal(win[:, 1], O.baked_windows(pts, sigma, ts, 5))
    # dense semantics where the dense tensor is affordable
    if n * ts[0] * ts[1] <= 8_000_000:
        d = O.splat_dense(pts, sigma, ts)
        s, o = R.splat_reduce(pts.cuda(), sigma, ts, num_std_sum=None, num_std_softor=None)
        close(s, O.reduce_sum(d))
        close(o, O.softor(d))


def test_edge_cases(R):
    ts = [40, 24]
    # points outside [0,1], on the borders, duplicates on a pixel centre (two exact-zero soft-OR factors), NaN
    pts = torch.tensor([[0.0, 0.0], [1.0, 1.0], [0.5, 0.5], [0.5, 0.5], [0.5, 0.5], [-0.2, 0.3], [1.4, 0.9], [0.25, 0.75],
                        [float("nan"), 0.5]])
    ok = pts[:8]
    s, o = R.splat_reduce(pts.cuda(), 9.0, ts, num_std_sum=None, num_std_softor=None)
    d = O.splat_dense(ok, 9.0, ts)
    close(s, O.reduce_sum(d))
    close(o, O.softor(d))
    wS = torch.randn(ts[1], ts[0], generator=torch.Generator().manual_seed(5))
    wO = torch.randn(ts[1], ts[0], generator=torch.Generator().manual_seed(6))
    p = ok.cuda().requires_grad_(True)
    s, o = R.splat_reduce(p, 9.0, ts, num_std_sum=None, num_std_softor=None)
    ((s * wS.cuda()).sum() + (o * wO.cuda()).sum()).backward()
    ana = O.splat_grad_analytic(ok, 9.0, ts, wS, wO, None, None)
    close_grad(p.grad, ana)
    assert torch.isfinite(p.grad).all()


@pytest.mark.parametrize("batched", [False, True])
def test_clustered_points_take_the_overflow_path(R, batched):
    """More than 16 candidates per 64x16 super tile: the warp-tile kernels hand those tiles to the overflow kernels."""
    gen = torch.Generator().manual_seed(11)
    n, ts, sigma = 120, [200, 136], 25.0
    pts = torch.cat([0.45 + 0.1 * torch.rand(90, 2, generator=gen), torch.rand(30, 2, generator=gen)])   # 90 points in a 20x14 texel patch
    wS, wO = torch.randn(ts[1], ts[0], generator=gen), torch.randn(ts[1], ts[0], generator=gen)
    if batched:
        p = pts.unsqueeze(0).repeat(3, 1, 1).cuda().requires_grad_(True)
        s, o = R.splat_reduce(p, sigma, ts)
        ((s * wS.cuda()).sum() + (o * wO.cuda()).sum()).backward()
        s, o, grad = s[2], o[2], p.grad[1]
    else:
        p = pts.cuda().requires_grad_(True)
        s, o = R.splat_reduce(p, sigma, ts)
        ((s * wS.cuda()).sum() + (o * wO.cuda()).sum()).backward()
        grad = p.grad
    close(s, O.baked_sum(pts, sigma, ts))
    close(o, O.baked_softor(pts, sigma, ts))
    ana = O.splat_grad_analytic(pts, sigma, ts, wS, wO, 4, 5)
    close_grad(grad, ana)
    # without the saved soft-OR output (first pass rebuilds the product)
    plan = R._SplatPlan(pts.cuda(), 1, sigma, ts[0], ts[1], 4, 5)
    d = plan.backward(pts.cuda(), wS.cuda().unsqueeze(0).contiguous(), wO.cuda().unsqueeze(0).contiguous(), False)
    close_grad(d[0], ana)


def _bin_padded(R, monkeypatch, pts, n_total, band, sigma, ts, gS, gO):
    """Forward and backward of `pts` padded to `n_total` points with points far off the texture (x = y = -5), appended after the
    real ones: their windows are empty, so they are never binned and the real points keep their indices -- every candidate list is
    the same, only N (and with it the binning kernel the library picks) changes.  Returns the sum and soft-OR textures and the
    gradients of the real points; the pad points' gradients must be exactly 0."""
    if band:
        monkeypatch.setenv("FFB_PREP_BAND_ROWS", band)
    else:
        monkeypatch.delenv("FFB_PREP_BAND_ROWS", raising=False)
    n = pts.shape[0]
    p = torch.cat([pts, torch.full((n_total - n, 2), -5.0)]).cuda()
    plan = R._SplatPlan(p, 1, sigma, ts[0], ts[1], 4, 5)
    s, o = plan.forward(p, True, True, False)
    d = plan.backward(p, gS, gO, False)
    assert torch.equal(d[:, n:], torch.zeros_like(d[:, n:]))
    return s.clone(), o.clone(), d[:, :n].clone()


@pytest.mark.parametrize("clustered", [False, True])
def test_binning_forms_agree_bitwise(R, monkeypatch, clustered):
    """The one-pass binning kernel (slot lists in shared memory, warp-wide entry stores; whole grid at once, or in bands of tile rows
    for grids that do not fit the shared arrays) and the count/scan/fill kernel that takes over when the one-pass kernel's shared
    arrays do not fit order every candidate list by point index, so the outputs are identical to the bit -- also with overflowing
    lists and with a tile count that is not a multiple of four (shared-memory rows stay 16-byte aligned)."""
    gen = torch.Generator().manual_seed(5)
    ts, sigma = ([200, 136] if clustered else [328, 200]), 25.0
    pts = torch.rand(400, 2, generator=gen)
    if clustered:
        pts[:150] = 0.45 + 0.1 * pts[:150]
    gS, gO = torch.randn(1, ts[1], ts[0], generator=gen).cuda(), torch.randn(1, ts[1], ts[0], generator=gen).cuda()
    # the one-pass kernel needs 40 B per super tile of a band + 16 N B of shared memory (WCH = 16 uint16 slots, two int counters)
    # within 226 KB, and N <= 65535: one tile row of these grids (6 or 4 super tiles) fits up to about 14,400 points
    forms = ((400, None),       # one-pass, whole grid
             (400, "3"),        # one-pass in bands of 3 tile rows
             (15000, None),     # count / scan / fill: 16 * 15000 B = 234 KB of records alone exceed 226 KB
             (70000, None))     # count / scan / fill: beyond the uint16 slot indices
    res = [_bin_padded(R, monkeypatch, pts, n, band, sigma, ts, gS, gO) for n, band in forms]
    for other in res[1:]:
        assert torch.equal(res[0][0], other[0]) and torch.equal(res[0][1], other[1])
        # the per-point gradient is a sum of per-tile partials added with float atomics: same terms, arrival order not fixed
        assert (res[0][2] - other[2]).norm() <= 1e-6 * other[2].norm()
    close(res[0][0][0], O.baked_sum(pts, sigma, ts))


def test_large_grid_takes_the_banded_binning(R, monkeypatch):
    """4096 x 2048 texels = 8192 super tiles: more than the one-pass binning kernel holds in shared memory at once, so it bins in
    bands of tile rows (chosen by the library).  Outputs identical to the count / scan / fill kernel's (the same points padded past
    what the one-pass kernel holds), which the smaller cases pin against the oracle; column sums of the sum texture against the
    closed form for a few points."""
    gen = torch.Generator().manual_seed(19)
    ts, sigma = [4096, 2048], 100.0
    pts = (torch.rand(1500, 2, generator=gen) * 0.98 + 0.01)
    gS, gO = torch.randn(1, ts[1], ts[0], generator=gen).cuda(), torch.randn(1, ts[1], ts[0], generator=gen).cuda()
    # one-pass shared memory: 40 B per super tile of a band + 16 N B within 226 KB; one tile row (64 super tiles, 2.5 KB) leaves
    # room for about 14,300 points, so 15,000 take count / scan / fill
    res = [_bin_padded(R, monkeypatch, pts, n, None, sigma, ts, gS, gO) for n in (1500, 15000)]
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    assert (res[0][2] - res[1][2]).norm() <= 1e-6 * res[1][2].norm()
    assert float(res[0][0].sum()) > 0 and torch.isfinite(res[0][2]).all()
    # one check against the closed form (fp64) on a crop: the 64 x 64 texels around the first point, sum texture with its windows
    P = pts[0] * torch.tensor([ts[0], ts[1]], dtype=torch.float32)
    c0, r0 = int(P[0]) - 32, int(P[1]) - 32
    c0, r0 = max(0, min(c0, ts[0] - 64)), max(0, min(r0, ts[1] - 64))
    near = ((pts * torch.tensor([ts[0], ts[1]], dtype=torch.float32) - P).abs().max(dim=1).values < 120)
    cols = torch.arange(c0, c0 + 64, dtype=torch.float64).view(1, 1, -1)
    rows = torch.arange(r0, r0 + 64, dtype=torch.float64).view(1, -1, 1)
    Pn = (pts[near].float() * torch.tensor([ts[0], ts[1]], dtype=torch.float32)).double()
    u = ((cols - Pn[:, 0].view(-1, 1, 1)) ** 2 + (rows - Pn[:, 1].view(-1, 1, 1)) ** 2) / sigma
    g = torch.exp(-u * u)
    H = O.footprint_size(sigma, 4)[1]
    f0 = torch.floor(Pn[:, 0].float() - H).double().view(-1, 1, 1) + H
    f1 = torch.floor(Pn[:, 1].float() - H).double().view(-1, 1, 1) + H
    inside = ((cols - f0).abs() <= H) & ((rows - f1).abs() <= H)
    want = (g * inside).sum(0).float()
    close(res[0][0][0, r0:r0 + 64, c0:c0 + 64].cpu(), want)


def test_saturated_softor_backward(R):
    """220 points inside a 20x20 texel patch at sigma = 100: the soft-OR saturates (prod(1 - g) runs from 1e-40 to 1e-2 across the
    patch), every super tile overflows.  The production backward rebuilds the product like torch.prod's backward.  A soft-OR window
    tighter than its no-op radius (num_std 2) takes the round-1 kernel, which reads the forward's output back when it is given
    (prod = 1 - O, an fp32 difference that loses the product's bits where O -> 1) and rebuilds the product otherwise.  All against
    the fp64 closed form, per component."""
    gen = torch.Generator().manual_seed(21)
    ts, sigma = [160, 160], 100.0
    pts = torch.cat([(70.0 + 20.0 * torch.rand(220, 2, generator=gen)) / 160.0, torch.rand(24, 2, generator=gen)])
    wS, wO = torch.randn(ts[1], ts[0], generator=gen), torch.randn(ts[1], ts[0], generator=gen)
    gs, go = wS.cuda().unsqueeze(0).contiguous(), wO.cuda().unsqueeze(0).contiguous()
    p1 = pts.cuda().unsqueeze(0).contiguous()
    for no in (5, 2):                                                          # exact soft-OR window / masked (round-1 kernel)
        ana = O.splat_grad_analytic(pts, sigma, ts, wS, wO, 4, no)
        so = O.baked_softor(pts, sigma, ts, num_std=no)
        assert float((1 - so).min()) < 1e-6 and float(so.max()) == 1.0        # the case does saturate
        plan = R._SplatPlan(p1, 1, sigma, ts[0], ts[1], 4, no)
        s, o = plan.forward(p1, True, True, False)
        close(o[0], so)
        close_grad(plan.backward(p1, gs, go, False, o)[0], ana)                # saved output (ignored by the production kernel)
        close_grad(plan.backward(p1, gs, go, False)[0], ana)                   # product rebuilt
    # a milder pattern where no list overflows (the main kernels, not the overflow kernels, see the saturation)
    gen = torch.Generator().manual_seed(22)
    pts2 = torch.cat([(40.0 + 80.0 * torch.rand(14, 2, generator=gen)) / 160.0 for _ in range(1)] + [(78.0 + 4.0 * torch.rand(2, 2, generator=gen)) / 160.0])
    pts2 = torch.cat([pts2, pts2[:8] + 0.004])                                 # near-coincident pairs: 1 - g small where it matters
    q1 = pts2.cuda().unsqueeze(0).contiguous()
    for no in (5, 2):
        ana2 = O.splat_grad_analytic(pts2, 400.0, ts, wS, wO, 4, no)
        plan2 = R._SplatPlan(q1, 1, 400.0, ts[0], ts[1], 4, no)
        _, o2 = plan2.forward(q1, True, True, False)
        close_grad(plan2.backward(q1, gs, go, False, o2)[0], ana2)
        close_grad(plan2.backward(q1, gs, go, False)[0], ana2)


def test_batched_and_shared_patterns(R):
    gen = torch.Generator().manual_seed(9)
    B, n, ts, sigma = 5, 40, [96, 72], 16.0
    pts = torch.rand(B, n, 2, generator=gen)
    gS, gO = torch.randn(B, ts[0], ts[1], generator=gen), torch.randn(B, ts[1], ts[0], generator=gen)
    p = pts.cuda().requires_grad_(True)
    s, o = R.splat_reduce(p, sigma, ts, sum_transposed=True)
    assert s.shape == (B, ts[0], ts[1]) and o.shape == (B, ts[1], ts[0])
    ((s * gS.cuda()).sum() + (o * gO.cuda()).sum()).backward()
    for b in range(B):
        close(s[b], O.baked_sum(pts[b], sigma, ts, transposed=True))
        close(o[b], O.baked_softor(pts[b], sigma, ts))
        ana = O.splat_grad_analytic(pts[b], sigma, ts, gS[b].T, gO[b], 4, 5)
        close_grad(p.grad[b], ana)
    # one pattern shared by all samples: gradient = sum over samples (linearity)
    q = pts[0].cuda().requires_grad_(True)
    s2, o2 = R.splat_reduce(q, sigma, ts, sum_transposed=True, batch=B)
    assert torch.equal(s2[3], s[0]) and torch.equal(o2[1], o[0])
    ((s2 * gS.cuda()).sum() + (o2 * gO.cuda()).sum()).backward()
    ana = O.splat_grad_analytic(pts[0], sigma, ts, gS.sum(0).T, gO.sum(0), 4, 5)
    close_grad(q.grad, ana)


def test_full_size_properties(R):
    """BASELINE config 3 shape (4096 points, 2048^2), one sample: size-independent properties."""
    gen = torch.Generator().manual_seed(0)
    pts = (torch.rand(4096, 2, generator=gen) * 0.96 + 0.02).cuda()
    ts = [2048, 2048]
    s, o = R.splat_reduce(pts, 100.0, ts)
    # (1) transposed layout is exactly the transpose; (2) swapping x/y transposes the image
    st, _ = R.splat_reduce(pts, 100.0, ts, sum_transposed=True)
    assert torch.equal(st, s.T.contiguous())
    s_sw, o_sw = R.splat_reduce(pts.flip(1).contiguous(), 100.0, ts)
    close(s_sw, s.T, rtol=1e-6, atol=1e-6)
    close(o_sw, o.T, rtol=1e-6, atol=1e-6)
    # (3) linearity of the sum over disjoint point subsets; soft-OR composes as 1-(1-a)(1-b)
    sa, oa = R.splat_reduce(pts[:2048].contiguous(), 100.0, ts)
    sb, ob = R.splat_reduce(pts[2048:].contiguous(), 100.0, ts)
    close(sa + sb, s, rtol=1e-5, atol=1e-6)
    close(1 - (1 - oa) * (1 - ob), o, rtol=1e-5, atol=1e-6)
    # (4) bounds and mass: 0 <= softor <= 1, softor <= sum, total mass = N * per-point footprint mass
    assert o.min() >= 0 and o.max() <= 1 and bool((o <= s + 1e-6).all())
    one = R.splat_reduce(torch.tensor([[0.5, 0.5]]).cuda(), 100.0, ts)[0].double().sum()
    close(s.double().sum() / 4096, one, rtol=1e-4, atol=0)
    # (5) a random 64x64 crop against the oracle evaluated on that crop's candidate points
    d = O.baked_sum(pts.cpu(), 100.0, ts)
    close(s[1000:1064, 300:364], d[1000:1064, 300:364])
    # (5b) the whole 2048^2 textures and the gradient for random upstream weights against the oracle (its scatter form + autograd
    #      finish in about a second at this size)
    gen2 = torch.Generator().manual_seed(4)
    wS, wO = torch.randn(2048, 2048, generator=gen2), torch.randn(2048, 2048, generator=gen2)
    po = pts.cpu().clone().requires_grad_(True)
    So = O.baked_softor(po, 100.0, ts)
    Sd = O.baked_sum(po, 100.0, ts)
    close(s, Sd.detach()); close(o, So.detach())
    ((Sd * wS).sum() + (So * wO).sum()).backward()
    pc = pts.clone().requires_grad_(True)
    sc, oc = R.splat_reduce(pc, 100.0, ts)
    ((sc * wS.cuda()).sum() + (oc * wO.cuda()).sum()).backward()
    close_grad(pc.grad, po.grad)
    # (6) gradient of the total mass w.r.t. interior points vanishes (translation invariance)
    p = pts.clone().requires_grad_(True)
    R.splat_reduce(p, 100.0, ts, reduce=("sum",))[0].sum().backward()
    inner = ((pts > 0.05) & (pts < 0.95)).all(1)
    assert p.grad[inner].abs().max() < 5e-2      # vs O(1e3) individual terms (3e-5 of them): sub-pixel sampling ripple + fp32 rounding of the distances


# ---- fused L1(softor, sum) backward (ffb_splat_bwd_l1; rasterization.py:586-607 test_point_reg) ---------------------
def _l1_case(R, pts, sigma, ts, sum_t):
    """(loss, d_pts) of the fused kernel, of the unfused ABI path and of the oracle's autograd for per-sample points."""
    import ctypes as C
    from fireflies_b200 import _native as nat
    B, N = pts.shape[0], pts.shape[1]
    plan = R._SplatPlan(pts, B, sigma, ts[0], ts[1], 4, 5)
    s, o = plan.forward(pts, True, True, sum_t)
    fused = plan.backward_l1(pts, s, o, sum_t)
    assert fused is not None, "fused L1 backward refused a case it should cover"
    loss_f, d_f = fused
    loss_u = torch.empty(B, device="cuda")
    gs, go = torch.empty_like(s), torch.empty_like(o)
    nat.check(nat.lib().ffb_l1_loss_fwd_bwd(o.data_ptr(), s.data_ptr(), 0, B, ts[0], ts[1], loss_u.data_ptr(), go.data_ptr(),
                                            gs.data_ptr(), nat.stream()), "l1")
    d_u = plan.backward(pts, gs, go, sum_t, o)
    loss_o, d_o = [], []
    for b in range(B):
        p = pts[b].cpu().clone().requires_grad_(True)
        S = O.baked_sum(p, sigma, ts, transposed=sum_t)
        So = O.baked_softor(p, sigma, ts)
        l = O.l1_loss(So, S)
        l.backward()
        loss_o.append(l.detach()); d_o.append(p.grad)
    return (loss_f, d_f), (loss_u, d_u), (torch.stack(loss_o), torch.stack(d_o))


@pytest.mark.parametrize("ts,sum_t,N,sigma,cluster", [([256, 256], True, 300, 36.0, False), ([320, 192], False, 200, 36.0, False),
                                                       ([256, 256], True, 120, 100.0, True), ([260, 260], True, 150, 25.0, False)])
def test_fused_l1_backward(R, ts, sum_t, N, sigma, cluster):
    gen = torch.Generator().manual_seed(11)
    B = 3
    pts = torch.rand(B, N, 2, generator=gen) * 0.9 + 0.05
    if cluster:                                             # long candidate lists: the overflow kernels take those super tiles
        pts = 0.45 + 0.1 * torch.rand(B, N, 2, generator=gen)
    pts = pts.cuda()
    (lf, df), (lu, du), (lo, do) = _l1_case(R, pts, sigma, ts, sum_t)
    close(lf, lu, rtol=2e-6, atol=0)                        # same textures, same signs: only the summation order differs
    close(df, du, rtol=1e-4, atol=1e-5 * float(du.abs().max()))
    close(lf, lo, rtol=1e-5, atol=1e-9)
    close_grad(df, do)


def test_fused_l1_refuses_what_it_cannot_pair(R):
    pts = (torch.rand(2, 50, 2, generator=torch.Generator().manual_seed(1)) * 0.8 + 0.1).cuda()
    plan = R._SplatPlan(pts, 2, 36.0, 256, 192, 4, 5)
    s, o = plan.forward(pts, True, True, True)
    assert plan.backward_l1(pts, s, o, True) is None        # [192,256] vs [256,192]: no elementwise pairing
    plan = R._SplatPlan(pts, 2, 36.0, 254, 254, 4, 5)       # sides not multiples of 4: no TMA description
    s, o = plan.forward(pts, True, True, True)
    assert plan.backward_l1(pts, s, o, True) is None


@pytest.mark.parametrize("B,shape", [(1, (5, 2)), (7, (33, 2)), (37, (1000,)), (256, (4096, 2)), (100, (300, 256)), (9, (256, 260))])
def test_reduce_over_samples(R, B, shape):
    x = torch.randn((B,) + shape, generator=torch.Generator().manual_seed(B)).cuda()
    out = R.reduce_over_samples(x)
    assert out.shape == shape
    close(out, x.double().sum(0), rtol=1e-5, atol=1e-5)
    assert torch.equal(out, R.reduce_over_samples(x))       # fixed summation order


def test_tma_and_plain_kernels_agree(R, monkeypatch):
    """The TMA-fed / TMA-stored kernels are the production path; textures the TMA unit cannot describe (sides not
    multiples of 4) and FFB_SPLAT_NO_TMA=1 take the plain-load / plain-store kernels.  Same arithmetic: forward bit for bit."""
    gen = torch.Generator().manual_seed(21)
    pts = (torch.rand(3, 400, 2, generator=gen) * 0.96 + 0.02).cuda()
    ts, sigma = [320, 272], 49.0
    gS, gO = torch.randn(3, ts[0], ts[1], generator=gen).cuda(), torch.randn(3, ts[1], ts[0], generator=gen).cuda()
    plan = R._SplatPlan(pts, 3, sigma, ts[0], ts[1], 4, 5)
    s1, o1 = plan.forward(pts, True, True, True)
    d1 = plan.backward(pts, gS, gO, True, o1)
    monkeypatch.setenv("FFB_SPLAT_NO_TMA", "1")
    s2, o2 = plan.forward(pts, True, True, True)
    d2 = plan.backward(pts, gS, gO, True, o1)
    monkeypatch.delenv("FFB_SPLAT_NO_TMA")
    assert torch.equal(s1, s2) and torch.equal(o1, o2)
    close(d1, d2, rtol=1e-5, atol=1e-5 * float(d2.abs().max()))
    # odd sides: no tensor map possible, the plain kernels run on their own; checked against the oracle
    pts1 = pts[0, :60].contiguous()
    ts_odd = [101, 75]
    s, o = R.splat_reduce(pts1, 16.0, ts_odd)
    close(s, O.baked_sum(pts1.cpu(), 16.0, ts_odd)); close(o, O.baked_softor(pts1.cpu(), 16.0, ts_odd))
    p = pts1.clone().requires_grad_(True)
    w = torch.randn(ts_odd[1], ts_odd[0], generator=gen).cuda()
    s, o = R.splat_reduce(p, 16.0, ts_odd)
    ((s * w).sum() + (o * w).sum()).backward()
    po = pts1.cpu().clone().requires_grad_(True)
    ((O.baked_sum(po, 16.0, ts_odd) * w.cpu()).sum() + (O.baked_softor(po, 16.0, ts_odd) * w.cpu()).sum()).backward()
    close_grad(p.grad, po.grad)


def test_backward_launch_forms(R, monkeypatch):
    """The super-tile backward has two launch forms for given upstream gradients: chunks of 8 consecutive items per one-warp CTA
    (dense patterns, FFB_SPLAT_EAGER=1; 5 x 17 super tiles x 2 samples = 170 items leave a ragged last chunk) and one CTA per item
    (sparse patterns, FFB_SPLAT_EAGER=0).  The fused L1 loss mode always takes a third: resident warps claiming items from a work
    counter.  Each against the fp64 closed form."""
    gen = torch.Generator().manual_seed(77)
    B, ts, sigma = 2, [260, 260], 49.0
    pts = (torch.rand(B, 120, 2, generator=gen) * 0.96 + 0.02)
    gS, gO = torch.randn(B, ts[0], ts[1], generator=gen), torch.randn(B, ts[1], ts[0], generator=gen)
    plan = R._SplatPlan(pts.cuda(), B, sigma, ts[0], ts[1], 4, 5)
    s, o = plan.forward(pts.cuda(), True, True, True)
    ana, ana_l1, loss_ref = [], [], []
    for b in range(B):
        ana.append(O.splat_grad_analytic(pts[b], sigma, ts, gS[b].T, gO[b], 4, 5))
        diff = o[b].cpu() - s[b].cpu()                     # loss = mean |softor - sum (as stored)|, rasterization.py:589-599
        sg = torch.sign(diff) / diff.numel()
        ana_l1.append(O.splat_grad_analytic(pts[b], sigma, ts, (-sg).T, sg, 4, 5))
        loss_ref.append(diff.abs().double().mean())
    for eager in ("1", "0"):
        monkeypatch.setenv("FFB_SPLAT_EAGER", eager)       # whatever the density heuristic says
        d = plan.backward(pts.cuda(), gS.cuda(), gO.cuda(), True).cpu()
        fused = plan.backward_l1(pts.cuda(), s, o, True)
        assert fused is not None
        loss, dl = fused
        for b in range(B):
            close_grad(d[b], ana[b])
            close(loss[b].cpu(), loss_ref[b].float(), rtol=1e-5, atol=1e-7)
            close_grad(dl[b].cpu(), ana_l1[b])


@pytest.mark.parametrize("want", [("sum",), ("softor",), ("sum", "softor")])
@pytest.mark.parametrize("sum_t", [False, True])
def test_every_kernel_variant(R, want, sum_t):
    """Each template instantiation of the production kernels (sum only / soft-OR only / both, natural or transposed sum,
    backward with and without the saved soft-OR output) against the oracle, plus the dense-radius (num_std = None) windows."""
    gen = torch.Generator().manual_seed(33)
    B, N, ts, sigma = 2, 250, [288, 224], 36.0
    pts = (torch.rand(B, N, 2, generator=gen) * 0.98 + 0.01)
    wS = torch.randn(B, ts[0], ts[1], generator=gen) if sum_t else torch.randn(B, ts[1], ts[0], generator=gen)
    wO = torch.randn(B, ts[1], ts[0], generator=gen)
    ws, wo = "sum" in want, "softor" in want
    # baked footprints / dense semantics / a soft-OR window tighter than its no-op radius (MASK_O kernels) / a sum window whose truncation
    # matters (MSK super-tile kernels; also the sum-only backward of (3, 2))
    for ns, no in ((4, 5), (0, 0), (3, 2), (3, 5)):
        plan = R._SplatPlan(pts.cuda(), B, sigma, ts[0], ts[1], ns, no)
        s, o = plan.forward(pts.cuda(), ws, wo, sum_t)
        grads = []
        for saved in (None, o) if wo else (None,):
            grads.append(plan.backward(pts.cuda(), wS.cuda() if ws else None, wO.cuda() if wo else None, sum_t, saved))
        for b in range(B):
            p = pts[b].clone().requires_grad_(True)
            tot = 0.0
            if ws:
                S = O.baked_sum(p, sigma, ts, num_std=ns, transposed=sum_t) if ns else O.reduce_sum(O.splat_dense(p, sigma, ts))
                if not ns and sum_t:
                    S = S.T
                close(s[b], S.detach())
                tot = tot + (S * wS[b]).sum()
            if wo:
                So = O.baked_softor(p, sigma, ts, num_std=no) if no else O.softor(O.splat_dense(p, sigma, ts))
                close(o[b], So.detach())
                tot = tot + (So * wO[b]).sum()
            tot.backward()
            for g in grads:
                close_grad(g[b], p.grad)


def test_l1_loss_single_pair_matches_torch(R):
    """test_point_reg's loop through the reference-shaped API for ONE pattern: 2-D textures in, scalar loss out."""
    gen = torch.Generator().manual_seed(2)
    pts = (torch.rand(100, 2, generator=gen) * 0.8 + 0.1)
    p = pts.cuda().requires_grad_(True)
    s, o = R.splat_reduce(p, 100.0, [512, 512], sum_transposed=True)
    loss = R.l1_loss(o, s)
    assert loss.dim() == 0
    loss.backward()
    po = pts.clone().requires_grad_(True)
    lo = O.l1_loss(O.baked_softor(po, 100.0, [512, 512]), O.baked_sum(po, 100.0, [512, 512], transposed=True))
    lo.backward()
    close(loss, lo.detach(), rtol=1e-5, atol=1e-9)
    close_grad(p.grad, po.grad)
