"""GPU parity of the line and depth rasterisers (SURVEY.md 8(f) row 2) against the reference-generated fixture
(tests/golden/lines_depth.npz, oracle/make_golden.py) and the CPU oracle.  Tolerances as for the point splat:
forward 1e-5 relative (+1e-6 absolute), gradients 1e-4 relative to the largest component.  The shapes here are small;
tests/test_lines_ref_gpu.py checks the same kernels against fp64 across line counts, ragged textures, culling radii,
geometry edges and every kernel instantiation."""
import numpy as np
import pytest
import torch

from oracle import ff_oracle as O

pytestmark = pytest.mark.gpu


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


def test_lines_forward_fixture(R, golden):
    g = golden("lines_depth")
    close(R.rasterize_lines(T(g["kat3_lines"]).cuda(), 4.0, T(np.array([8, 6]))), g["kat3"])
    lines, ts, sig = T(g["lines"]).cuda(), g["lines_ts"].tolist(), float(g["lines_sigma"])
    keep = lines.clone()
    close(R.rasterize_lines(lines, sig, ts), g["lines_dense"])
    assert torch.equal(lines, keep)                          # documented deviation: the argument is not scaled in place
    s, o = R.lines_reduce(lines, sig, ts)
    close(s, g["lines_sum"]); close(o, g["lines_softor"])
    s2, none = R.lines_reduce(lines, sig, ts, reduce=("sum",))
    assert none is None and torch.equal(s2, s)


def test_lines_backward_fixture(R, golden):
    g = golden("lines_depth")
    ts, sig = g["lines_ts"].tolist(), float(g["lines_sigma"])
    wS, wO, ref = T(g["lines_wS"]).cuda(), T(g["lines_wO"]).cuda(), g["lines_weighted_grad"]
    tol = dict(rtol=1e-4, atol=1e-4 * np.abs(ref).max())
    l = T(g["lines"]).cuda().requires_grad_(True)            # dense tensor + torch reductions, like the reference
    tex = R.rasterize_lines(l, sig, ts)
    ((tex.sum(dim=0) * wS).sum() + (R.softor(tex) * wO).sum()).backward()
    close(l.grad, ref, **tol)
    l = T(g["lines"]).cuda().requires_grad_(True)            # fused reductions
    s, o = R.lines_reduce(l, sig, ts)
    ((s * wS).sum() + (o * wO).sum()).backward()
    close(l.grad, ref, **tol)
    l = T(g["lines"]).cuda().requires_grad_(True)            # test_line_reg's loss (rasterization.py:692-697)
    s, o = R.lines_reduce(l, sig, ts)
    loss = torch.nn.functional.l1_loss(o, s)
    loss.backward()
    close(loss, g["lines_l1"], rtol=1e-5, atol=1e-8)
    r1 = g["lines_l1_grad"]
    close(l.grad, r1, rtol=1e-4, atol=1e-4 * np.abs(r1).max())


def test_lines_on_texel_centres_and_larger_frame(R):
    """texels exactly on a line (g == 1: torch.prod's zero handling in the soft-OR backward), 512^2 like test_line_reg."""
    ts, sig = [512, 512], 10.0
    gen = torch.Generator().manual_seed(3)
    lines = torch.rand(50, 2, 2, generator=gen) * 0.8 + 0.1
    lines[0] = torch.tensor([[0.25, 0.5], [0.75, 0.5]])      # horizontal, through texel centres (row 256)
    lines[1] = torch.tensor([[0.5, 0.125], [0.5, 0.875]])    # vertical, crossing line 0 on a texel centre
    wS, wO = torch.randn(512, 512, generator=gen), torch.randn(512, 512, generator=gen)
    lo = lines.clone().requires_grad_(True)
    tex = O.rasterize_lines(lo, sig, ts)
    S, So = tex.sum(dim=0), O.softor(tex)
    ((S * wS).sum() + (So * wO).sum()).backward()
    l = lines.cuda().requires_grad_(True)
    s, o = R.lines_reduce(l, sig, ts)
    close(s, S); close(o, So)
    ((s * wS.cuda()).sum() + (o * wO.cuda()).sum()).backward()
    ref = lo.grad.numpy()
    close(l.grad, ref, rtol=1e-4, atol=1e-4 * np.abs(ref).max())


def test_depth_fixture_and_gradients(R, golden):
    g = golden("lines_depth")
    pts, ts, sig = T(g["depth_points"]), g["depth_ts"].tolist(), float(g["depth_sigma"])
    close(R.rasterize_depth(pts[:, 0:2].cuda(), pts[:, 2:3].cuda(), sig, T(np.array(ts))), g["depth_dense"])
    for i, lv in enumerate(R.subsampled_point_raster(pts.cuda(), 3, sig, ts)):
        close(lv, g[f"depth_level{i}"])
    # gradients w.r.t. points and depth against the oracle's autograd (points inside the frame, away from texel midpoints)
    gen = torch.Generator().manual_seed(9)
    p = (torch.rand(7, 2, generator=gen) * 0.8 + 0.1)
    d = torch.rand(7, 1, generator=gen) + 0.2
    w = torch.randn(7, ts[1], ts[0], generator=gen)
    po, do_ = p.clone().requires_grad_(True), d.clone().requires_grad_(True)
    (O.rasterize_depth(po, do_, sig, ts) * w).sum().backward()
    pc, dc = p.cuda().requires_grad_(True), d.cuda().requires_grad_(True)
    (R.rasterize_depth(pc, dc, sig, ts) * w.cuda()).sum().backward()
    close(pc.grad, po.grad, rtol=1e-4, atol=1e-4 * float(po.grad.abs().max()))
    close(dc.grad, do_.grad, rtol=1e-4, atol=1e-4 * float(do_.grad.abs().max()))


def test_epipolar_lines(R):
    import fireflies_b200 as ff
    Laser = ff.projection.Laser
    rays = Laser.generate_uniform_rays(0.02, 4, 4)
    K = ff.utils.io.build_projection_matrix(60, 0.01, 1000.0)
    laser = Laser(ff.entity.Transformable("projector"), rays, K, 60.0, 0.5, 5.0)
    cam = torch.eye(4, device="cuda"); cam[0, 3] = 0.3
    tex = laser.render_epipolar_lines(6.0, torch.tensor([64, 48]), camera_to_world=cam)
    assert tex.shape == (16, 48, 64)
    lo = laser.originPerRay() + 0.5 * laser.rays()
    hi = laser.originPerRay() + 5.0 * laser.rays()
    w2c = cam.inverse().cpu()
    Kc = K.cpu() if torch.is_tensor(K) else torch.as_tensor(K)
    lo2 = O.transform_points(O.transform_points(lo.cpu(), w2c), Kc.float())[:, 0:2]
    hi2 = O.transform_points(O.transform_points(hi.cpu(), w2c), Kc.float())[:, 0:2]
    close(tex, O.rasterize_lines(torch.stack([lo2, hi2], dim=1), 6.0, [64, 48]))


def test_points_in_texel_units(R, golden):
    """rasterize_points_in_non_ndc (rasterization.py:38-63), forward and gradient against reference-generated values."""
    g = golden("lines_depth")
    p = T(g["px_points"]).cuda().requires_grad_(True)
    tex = R.rasterize_points_in_non_ndc(p, 6.0, T(np.array([40, 24])))
    close(tex, g["px_dense"])
    (tex * T(g["px_w"]).cuda()).sum().backward()
    ref = g["px_grad"]
    close(p.grad, ref, rtol=1e-4, atol=1e-4 * np.abs(ref).max())
