"""GPU: the differentiable projector texture (main.py:64-77) -- the blur's adjoint kernel (ffb_blur_bwd), the differentiable
``gaussian_blur2d``, ``Laser.projector_texture`` and the batched ``TextureStep`` -- against torch autograd of the oracle's
restatement (reflect padding + conv2d; its autograd is the reference adjoint), the adjoint identity, and across two ranks.

Tolerances: forward 1e-5 relative + 1e-6 absolute; ray gradients 1e-4 of each ray's gradient norm, floored at a tenth of the
mean ray gradient norm (as the splat tests judge point gradients)."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import ff_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ff():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import fireflies_b200
    return fireflies_b200


def close(a, b, rtol=1e-5, atol=1e-6):
    a = a.detach().cpu().double().numpy() if torch.is_tensor(a) else np.asarray(a, np.float64)
    b = b.detach().cpu().double().numpy() if torch.is_tensor(b) else np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    err = np.abs(a - b) - (atol + rtol * np.abs(b))
    assert err.max() <= 0, f"max violation {err.max():.3e}; max abs diff {np.abs(a - b).max():.3e}"


def close_grad(got, ref, rtol=1e-4):
    """per component: |got - ref| <= rtol |ref| + rtol max(||ref[ray]||_2, 0.1 mean_m ||ref[m]||_2)."""
    a = got.detach().cpu().double().numpy()
    b = ref.detach().cpu().double().numpy()
    assert a.shape == b.shape, (a.shape, b.shape)
    nrm = np.linalg.norm(b, axis=-1, keepdims=True)
    scale = np.maximum(nrm, 0.1 * nrm.mean())
    err = np.abs(a - b) - (rtol * np.abs(b) + rtol * scale)
    assert err.max() <= 0, f"max violation {err.max():.3e}; max abs diff {np.abs(a - b).max():.3e}, mean norm {nrm.mean():.3e}"


def oracle_blur_grad(x, g, ks, sg):
    xr = x.detach().cpu().clone().requires_grad_(True)
    O.gaussian_blur2d(xr, ks, sg).backward(g.detach().cpu())
    return xr.grad


BLUR_CASES = [
    ((2, 3, 64, 128), (3, 3), (1.5, 1.5)),      # sliding-window adjoint, k = 3, 5, 11
    ((2, 3, 64, 128), (5, 5), (3.0, 3.0)),
    ((2, 3, 64, 128), (11, 11), (5.0, 5.0)),
    ((2, 3, 37, 50), (5, 5), (3.0, 3.0)),       # W % 4 != 0: generic
    ((2, 3, 64, 128), (7, 7), (2.0, 2.0)),      # generic sizes
    ((2, 3, 64, 128), (5, 3), (3.0, 1.5)),      # anisotropic
    ((2, 3, 6, 12), (11, 11), (5.0, 5.0)),      # h = 5: both folds hit the same texels
    ((2, 3, 64, 64), (11, 11), (2.0, 4.0)),     # sliding window, anisotropic sigma, one tile wide
]


@pytest.mark.parametrize("shape,ks,sg", BLUR_CASES)
def test_blur_backward_vs_oracle_autograd(ff, shape, ks, sg):
    gen = torch.Generator().manual_seed(11)
    x, g = torch.rand(shape, generator=gen), torch.randn(shape, generator=gen)
    xc = x.cuda().requires_grad_(True)
    y = ff.postprocessing.gaussian_blur2d(xc, ks, sg)
    close(y, O.gaussian_blur2d(x, ks, sg))
    y.backward(g.cuda())
    close(xc.grad, oracle_blur_grad(x, g, ks, sg))


def test_blur_backward_unaligned_storage(ff):
    """The sliding-window conditions hold except for a pointer one element into its buffer: the plain-load kernels run."""
    from fireflies_b200.postprocessing.gauss_blur import gaussian_blur2d_backward
    shape, ks, sg = (2, 3, 64, 128), (5, 5), (3.0, 3.0)
    n = int(np.prod(shape))
    gen = torch.Generator().manual_seed(12)
    xb, gb = torch.rand(n + 1, generator=gen).cuda(), torch.randn(n + 1, generator=gen).cuda()
    x, g = xb[1:].view(shape), gb[1:].view(shape)
    assert x.data_ptr() % 16 != 0 and g.data_ptr() % 16 != 0
    ref = oracle_blur_grad(x, g, ks, sg)
    close(gaussian_blur2d_backward(g, ks, sg), ref)
    xa = xb[1:].view(shape).detach().requires_grad_(True)    # a leaf on the unaligned storage
    ff.postprocessing.gaussian_blur2d(xa, ks, sg).backward(g)
    close(xa.grad, ref)


@pytest.mark.parametrize("k", [3, 5, 11])
def test_adjoint_identity(ff, k):
    """<blur(x), g> == <x, blur_bwd(g)> in fp64 sums: catches any fold error at the borders independently of the oracle."""
    from fireflies_b200.postprocessing.base import run_postprocess
    from fireflies_b200.postprocessing.gauss_blur import gaussian_blur2d_backward
    gen = torch.Generator(device="cuda").manual_seed(k)
    x = torch.rand((4, 1024, 1024), device="cuda", generator=gen)
    g = torch.rand((4, 1024, 1024), device="cuda", generator=gen)
    spec = ((k, k), (k / 2.0, k / 2.0))
    lhs = (run_postprocess(x, blur=spec).double() * g.double()).sum()
    rhs = (x.double() * gaussian_blur2d_backward(g, *spec).double()).sum()
    assert abs(float(lhs - rhs)) <= 1e-6 * abs(float(lhs)), (float(lhs), float(rhs))


@pytest.mark.parametrize("shape,ks,sg", [((2, 3, 64, 128), (5, 5), (3.0, 3.0)), ((1, 2, 37, 50), (3, 5), (1.0, 2.0)),
                                         ((1, 1, 500, 500), 11, 5.0)])
def test_gaussian_blur2d_forward_is_run_postprocess(ff, shape, ks, sg):
    from fireflies_b200.postprocessing.base import run_postprocess
    from fireflies_b200.postprocessing.gauss_blur import blur_spec
    x = torch.rand(shape, generator=torch.Generator().manual_seed(3)).cuda()
    got = ff.postprocessing.gaussian_blur2d(x, ks, sg)
    want = run_postprocess(x.reshape(-1, shape[-2], shape[-1]), blur=blur_spec(ks, sg)).view(shape)
    assert torch.equal(got, want)


# ---- the projector texture ---------------------------------------------------------------------------------------------
_A01 = torch.tensor([[0.5, 0.0, 0.0, 0.5], [0.0, 0.5, 0.0, 0.5], [0.0, 0.0, 1.0, 0.0], [0.0, 0.0, 0.0, 1.0]])


def perspective01():
    """NDC x, y -> 0.5 x + 0.5 (homogeneous): the projected rays land in [0, 1] as the splat expects."""
    return _A01 @ O.build_projection_matrix(60, 0.01, 1000.0)


def make_laser(ff, rays, device="cuda"):
    return ff.projection.Laser(ff.entity.Transformable("projector"), rays.to(device), perspective01().to(device), 60.0, 0.01, 1000.0)


def oracle_texture(rays, sigma, ts, blur, points=None):
    """The oracle composition; ``points`` (the projected rays' xy) replaces its first stage when given."""
    if points is None:
        points = O.rays_to_ndc(rays, perspective01())[:, 0:2]
    tex = O.reduce_sum(O.splat_dense(points, sigma, ts))
    if blur is not None:
        tex = O.gaussian_blur2d(tex, *blur)
    zero = torch.zeros_like(tex)
    return torch.stack([zero, tex, zero]).movedim(0, -1)


def oracle_ray_grad(rays, sigma, ts, blur, w):
    r = rays.detach().cpu().clone().requires_grad_(True)
    (oracle_texture(r, sigma, ts, blur) * w.cpu()).sum().backward()
    return r.grad


BLUR = ((5, 5), (3.0, 3.0))


def check_texture_forward(laser, tex, rays, sigma, ts, blur):
    """The forward against the oracle composition, split at its projection.  With the [0, 1] remap folded into the perspective
    a projected coordinate is a sum of two products, and the device's fused multiply-adds and torch's CPU matmul round it
    differently in the last bit (either is as far from the fp64 projection as the other).  At sigma 10 a texel value moves
    by up to ~0.5 per texel of point shift, so one ulp of a coordinate times 500 texels (3e-5 texels) moves the texture by up
    to 9e-6: more than the forward tolerance allows.  So the projection is held to 4 ulps of the oracle's (the two roundings
    of the homogeneous coordinate and the division's give up to 2 at this shape), and the splat + blur + stack to the forward
    tolerance on the points the device projected."""
    pts = laser.projectRaysToNDC()[:, 0:2].detach().cpu()
    ref_pts = O.rays_to_ndc(rays, perspective01())[:, 0:2]
    ulp = torch.from_numpy(np.spacing(torch.maximum(pts.abs(), ref_pts.abs()).numpy()))
    assert (pts - ref_pts).abs().le(4 * ulp).all(), float(((pts - ref_pts).abs() / ulp).max())
    close(tex, oracle_texture(rays, sigma, ts, blur, points=pts))


def test_projector_texture_config1_forward(ff):
    """configs[1]: 18x18 uniform rays (0.0275), 500^2, sigma 10, (5,5)/(3,3) blur -- the full-size texture."""
    rays = O.uniform_rays(0.0275, 18, 18)
    laser = make_laser(ff, rays)
    tex = laser.projector_texture(10.0, [500, 500], blur=BLUR)
    assert tex.shape == (500, 500, 3)
    check_texture_forward(laser, tex, rays, 10.0, [500, 500], BLUR)


@pytest.mark.parametrize("ts", [[128, 96], [96, 96]])
def test_projector_texture_gradient(ff, ts):
    """d (tex * Wt).sum() / d rays against torch autograd of the oracle composition (8x8 rays; 128x96 catches orientation
    mistakes)."""
    rays = O.uniform_rays(0.06, 8, 8)
    w = torch.randn((ts[1], ts[0], 3), generator=torch.Generator().manual_seed(4))
    laser = make_laser(ff, rays)
    laser._rays.requires_grad_(True)
    tex = laser.projector_texture(10.0, ts, blur=BLUR)
    check_texture_forward(laser, tex, rays, 10.0, ts, BLUR)
    (tex * w.cuda()).sum().backward()
    close_grad(laser._rays.grad, oracle_ray_grad(rays, 10.0, ts, BLUR, w))


def test_projector_texture_without_blur(ff):
    rays = O.uniform_rays(0.06, 8, 8)
    w = torch.randn((96, 128, 3), generator=torch.Generator().manual_seed(5))
    laser = make_laser(ff, rays)
    laser._rays.requires_grad_(True)
    tex = laser.projector_texture(10.0, [128, 96], blur=None)
    check_texture_forward(laser, tex, rays, 10.0, [128, 96], None)
    (tex * w.cuda()).sum().backward()
    close_grad(laser._rays.grad, oracle_ray_grad(rays, 10.0, [128, 96], None, w))


# ---- TextureStep ---------------------------------------------------------------------------------------------------------
def autograd_ray_grad(ff, rays, sigma, ts, blur, g_sum):
    laser = make_laser(ff, rays)
    laser._rays.requires_grad_(True)
    (laser.projector_texture(sigma, ts, blur=blur) * g_sum).sum().backward()
    return laser._rays.grad


@pytest.mark.parametrize("ts,blur", [([128, 96], BLUR), ([96, 96], ((11, 11), (5.0, 5.0))), ([128, 96], None),
                                     ([500, 500], BLUR)])
def test_texture_step_matches_autograd(ff, ts, blur):
    rays = O.uniform_rays(0.06, 8, 8) if ts[0] < 500 else O.uniform_rays(0.0275, 18, 18)
    g = torch.randn((8, ts[1], ts[0], 3), generator=torch.Generator().manual_seed(6)).cuda()
    laser = make_laser(ff, rays)
    laser._rays.requires_grad_(True)
    step = ff.TextureStep(laser, sigma=10.0, texture_size=ts, blur=blur)
    tex = step.texture()
    assert torch.equal(tex, laser.projector_texture(10.0, ts, blur=blur).detach())
    ref = autograd_ray_grad(ff, rays, 10.0, ts, blur, g.sum(0))
    d = step.backward(g).clone()
    close_grad(d, ref)
    assert torch.equal(laser._rays.grad, d)
    d2 = step.backward(g)                                      # a second call accumulates like autograd
    close_grad(d2, d, rtol=1e-5)                               # the splat backward sums into d_pts with float atomics
    assert torch.equal(laser._rays.grad, d + d2)


def test_texture_step_single_sample_and_ignored_channels(ff):
    """The splat backward sums into d_pts with float atomics, so repeated calls agree to rounding, not bitwise."""
    ts = [128, 96]
    rays = O.uniform_rays(0.06, 8, 8)
    g = torch.randn((1, ts[1], ts[0], 3), generator=torch.Generator().manual_seed(7)).cuda()
    laser = make_laser(ff, rays)
    step = ff.TextureStep(laser, sigma=10.0, texture_size=ts, blur=BLUR)
    step.texture()
    d_b1 = step.backward(g).clone()
    d_hw3 = step.backward(g[0]).clone()
    close_grad(d_hw3, d_b1, rtol=1e-5)
    g2 = g.clone()
    g2[..., 0] = 123.0
    g2[..., 2] = torch.randn_like(g2[..., 2])
    close_grad(step.backward(g2), d_b1, rtol=1e-5)              # channels 0 and 2 multiply constants
    B8 = torch.randn((8, ts[1], ts[0], 3), device="cuda")
    d8 = step.backward(B8).clone()
    B8c = B8.clone()
    B8c[..., 0::2] = torch.randn_like(B8c[..., 0::2])
    close_grad(step.backward(B8c), d8, rtol=1e-5)


# ---- two ranks -----------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        _rank_checks(rank, world, dev)
    except BaseException:  # noqa: BLE001  (a failing rank must not wait for its peers in destroy_process_group: leave at once)
        import traceback
        traceback.print_exc()
        os._exit(1)
    dist.destroy_process_group()


def _rank_checks(rank, world, dev):
    import torch.distributed as dist
    import fireflies_b200 as ff
    singles = [dist.new_group([r]) for r in range(world)]       # every rank creates every group, in the same order
    ts, B = [500, 500], 8 * world
    rays = O.uniform_rays(0.0275, 18, 18)
    g = torch.randn((B, ts[1], ts[0], 3), generator=torch.Generator().manual_seed(9)).to(dev)
    sharded = ff.TextureStep(make_laser(ff, rays, dev), sigma=10.0, texture_size=ts, blur=BLUR)
    sharded.texture()
    d = sharded.backward(g[rank::world]).clone()
    full = ff.TextureStep(make_laser(ff, rays, dev), sigma=10.0, texture_size=ts, blur=BLUR, process_group=singles[rank])
    full.texture()
    ref = full.backward(g).clone()
    close_grad(d, ref, rtol=1e-5)
    gathered = [torch.empty_like(d) for _ in range(world)]
    dist.all_gather(gathered, d)
    assert all(torch.equal(x, gathered[0]) for x in gathered)
    torch.cuda.synchronize()


def test_texture_step_two_ranks(ff):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port()), nprocs=2, join=True)
