"""GPU: gradients of ``transform_points`` / ``transform_directions`` w.r.t. the 4x4 matrix (``ffb_transform_points_bwd_full``)
and what they make differentiable -- the projector texture w.r.t. ``Laser._perspective``, the epipolar lines w.r.t. the camera
pose, and ``TextureStep`` with a perspective that requires grad.

Tolerances: d_T against the fp64 closed form per entry ``1e-5 * sum_v |d_i p~_j|`` (entries can cancel); against torch autograd
of the oracle, ``close_grad`` at 1e-4 as in test_texture_gpu.py.  A matrix gradient through the splat is a sum over rays of
each ray's term, so it is held to the error the ray-gradient tolerance allows in every term (``oracle_k_grad``)."""
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
    """per component: |got - ref| <= rtol |ref| + rtol max(||ref[row]||_2, 0.1 mean ||ref[m]||_2)."""
    a = got.detach().cpu().double().numpy()
    b = ref.detach().cpu().double().numpy()
    assert a.shape == b.shape, (a.shape, b.shape)
    nrm = np.linalg.norm(b, axis=-1, keepdims=True)
    scale = np.maximum(nrm, 0.1 * nrm.mean())
    err = np.abs(a - b) - (rtol * np.abs(b) + rtol * scale)
    assert err.max() <= 0, f"max violation {err.max():.3e}; max abs diff {np.abs(a - b).max():.3e}, mean norm {nrm.mean():.3e}"


def within(got, ref, scale, rtol):
    a, b = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    err = np.abs(a - b) - rtol * np.asarray(scale, np.float64)
    assert err.max() <= 0, f"max violation {err.max():.3e}; |diff| {np.abs(a - b).max():.3e}; scale {np.asarray(scale).max():.3e}"


# ---- the entry point against the fp64 closed form ------------------------------------------------------------------------
def rigid_world():
    a, b = 0.7, -0.4
    Rz = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
    Rx = np.array([[1, 0, 0], [0, np.cos(b), -np.sin(b)], [0, np.sin(b), np.cos(b)]])
    W = np.eye(4)
    W[:3, :3], W[:3, 3] = Rz @ Rx, [0.3, -1.2, 2.5]
    return W.astype(np.float32)


def transforms(golden, rng):
    A = np.eye(4, dtype=np.float32)
    A[:3] = rng.standard_normal((3, 4)).astype(np.float32)
    return {"tp_K": golden("transforms")["tp_K"], "rigid": rigid_world(), "affine": A}


def points_and_grads(V, seed):
    """N(0,1) x, y and g; z in [-5, -1] so the projective tp_K (w = -z) stays away from w = 0."""
    rng = np.random.default_rng(seed)
    p = rng.standard_normal((V, 3)).astype(np.float32)
    p[:, 2] = -(1.0 + 4.0 * rng.random(V)).astype(np.float32)
    return p, rng.standard_normal((V, 3)).astype(np.float32), rng


def closed_form(p, T, g, dirs):
    """fp64 d_T = sum_v d(v) p~(v)^T and the per-entry sum of |terms|."""
    p, T, g = p.astype(np.float64), T.astype(np.float64), g.astype(np.float64)
    pt = np.hstack([p, np.full((len(p), 1), 0.0 if dirs else 1.0)])
    if dirs:
        d = np.hstack([g, np.zeros((len(p), 1))])
    else:
        h = pt @ T.T
        inv = 1.0 / h[:, 3]
        d = np.hstack([g * inv[:, None], (-(g * h[:, :3]).sum(1) * inv * inv)[:, None]])
    return d.T @ pt, np.abs(d).T @ np.abs(pt)


def full_bwd(ff, pts, T, g, dirs, want_pts=True):
    """ffb_transform_points_bwd_full on device tensors -> (d_pts or None, d_T [4,4])."""
    L = ff._native.lib()
    V = pts.shape[0]
    d = torch.empty_like(pts) if want_pts else None
    dT = torch.empty(16, dtype=torch.float32, device="cuda")
    nb = L.ffb_transform_bwd_workspace_bytes(V)
    ws = torch.empty(max(nb, 1), dtype=torch.uint8, device="cuda")
    rc = L.ffb_transform_points_bwd_full(pts.data_ptr(), V, T.data_ptr(), int(dirs), g.data_ptr(), None if d is None else d.data_ptr(),
                                         dT.data_ptr(), ws.data_ptr() if nb else None, nb, torch.cuda.current_stream().cuda_stream)
    assert rc == 0, L.ffb_last_error_string()
    return d, dT.view(4, 4)


def points_bwd(ff, pts, T, g, dirs):
    d = torch.empty_like(pts)
    rc = ff._native.lib().ffb_transform_points_bwd(pts.data_ptr(), pts.shape[0], T.data_ptr(), int(dirs), g.data_ptr(), d.data_ptr(),
                                                   torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    return d


SIZES = [1, 3, 4, 5, 1023, 1024, 1025, 4099, 2 ** 20, 3 * 10 ** 6 + 1]


@pytest.mark.parametrize("dirs", [False, True], ids=["points", "directions"])
@pytest.mark.parametrize("V", SIZES)
def test_d_transform_against_closed_form(ff, golden, V, dirs):
    """Every transform, both layouts of work (one CTA / partials + fold), with and without d_pts: d_T within the summed
    tolerance, d_T identical with and without d_pts and across calls, d_pts identical to ffb_transform_points_bwd."""
    p, g, rng = points_and_grads(V, V)
    pc, gc = torch.from_numpy(p).cuda(), torch.from_numpy(g).cuda()
    for name, T in transforms(golden, rng).items():
        Tc = torch.from_numpy(T).cuda()
        ref, scale = closed_form(p, T, g, dirs)
        d_pts, dT = full_bwd(ff, pc, Tc, gc, dirs)
        within(dT.cpu().numpy(), ref, scale, 1e-5)
        if dirs:
            assert (dT[3] == 0).all() and (dT[:, 3] == 0).all(), name
        assert torch.equal(d_pts, points_bwd(ff, pc, Tc, gc, dirs)), name
        none, dT_only = full_bwd(ff, pc, Tc, gc, dirs, want_pts=False)
        assert none is None and torch.equal(dT_only, dT), name
        assert torch.equal(full_bwd(ff, pc, Tc, gc, dirs)[1], dT), name


def test_zero_points_write_zeros(ff):
    buf = torch.zeros((1, 3), device="cuda")
    T = torch.eye(4, device="cuda")
    dT = torch.full((16,), 7.0, device="cuda")
    L = ff._native.lib()
    assert L.ffb_transform_bwd_workspace_bytes(0) == 0
    assert L.ffb_transform_points_bwd_full(buf.data_ptr(), 0, T.data_ptr(), 0, buf.data_ptr(), None, dT.data_ptr(), None, 0,
                                           torch.cuda.current_stream().cuda_stream) == 0
    assert (dT == 0).all()


# ---- autograd against the oracle -----------------------------------------------------------------------------------------
def oracle_grads(p, K, w, dirs, need_p, need_K):
    pr = p.clone().requires_grad_(need_p)
    Kr = K.clone().requires_grad_(need_K)
    f = O.transform_directions if dirs else O.transform_points
    (f(pr, Kr) * w).sum().backward()
    return pr.grad, Kr.grad


@pytest.mark.parametrize("dirs", [False, True], ids=["points", "directions"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_autograd_matrix_only(ff, golden, dirs, dtype):
    p, _, _ = points_and_grads(4099, 1)
    p = torch.from_numpy(p)
    K = torch.from_numpy(golden("transforms")["tp_K"]).to(dtype)
    w = torch.randn((p.shape[0], 3), generator=torch.Generator().manual_seed(2))
    Kc = K.cuda().requires_grad_(True)
    pc = p.cuda()
    f = ff.utils.math.transform_directions if dirs else ff.utils.math.transform_points
    (f(pc, Kc) * w.cuda()).sum().backward()
    _, ref = oracle_grads(p, K, w, dirs, False, True)
    assert Kc.grad.dtype == dtype and Kc.grad.shape == (4, 4)
    close_grad(Kc.grad, ref)


@pytest.mark.parametrize("dirs", [False, True], ids=["points", "directions"])
def test_autograd_points_only_is_the_points_kernel(ff, golden, dirs):
    """Only the points require grad: the gradient is the points-only kernel's, bit for bit."""
    p, _, _ = points_and_grads(1025, 3)
    p = torch.from_numpy(p)
    K = torch.from_numpy(golden("transforms")["tp_K"])
    w = torch.randn((p.shape[0], 3), generator=torch.Generator().manual_seed(4))
    pc = p.cuda().requires_grad_(True)
    f = ff.utils.math.transform_directions if dirs else ff.utils.math.transform_points
    (f(pc, K.cuda()) * w.cuda()).sum().backward()
    assert torch.equal(pc.grad, points_bwd(ff, p.cuda(), K.cuda(), w.cuda(), dirs))
    ref, _ = oracle_grads(p, K, w, dirs, True, False)
    close_grad(pc.grad, ref)


def test_autograd_points_and_matrix(ff, golden):
    p, _, _ = points_and_grads(4099, 5)
    p = torch.from_numpy(p)
    K = torch.from_numpy(golden("transforms")["tp_K"])
    w = torch.randn((p.shape[0], 3), generator=torch.Generator().manual_seed(6))
    pc, Kc = p.cuda().requires_grad_(True), K.cuda().requires_grad_(True)
    (ff.utils.math.transform_points(pc, Kc) * w.cuda()).sum().backward()
    rp, rK = oracle_grads(p, K, w, False, True, True)
    close_grad(pc.grad, rp)
    close_grad(Kc.grad, rK)
    assert torch.equal(pc.grad, points_bwd(ff, p.cuda(), K.cuda(), w.cuda(), False))


def test_double_backward_is_refused(ff, golden):
    K = torch.from_numpy(golden("transforms")["tp_K"]).cuda().requires_grad_(True)
    p = torch.from_numpy(points_and_grads(8, 7)[0]).cuda()
    out = ff.utils.math.transform_points(p, K)
    (gK,) = torch.autograd.grad(out, K, torch.ones_like(out, requires_grad=True), create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable"):
        gK.sum().backward()


def test_storage_edges(ff, golden):
    """Points 12 bytes into their storage (scalar loads) and a non-contiguous upstream gradient: same bits as the aligned,
    contiguous call."""
    V = 4099
    p, g, _ = points_and_grads(V, 8)
    K = torch.from_numpy(golden("transforms")["tp_K"]).cuda()
    buf = torch.zeros((V + 1, 3), device="cuda")
    buf[1:] = torch.from_numpy(p).cuda()
    pv = buf[1:]
    assert pv.is_contiguous() and pv.data_ptr() % 16 == 12
    g_nc = torch.from_numpy(np.ascontiguousarray(g.T)).cuda().t()          # [V, 3] view of a [3, V] tensor
    assert not g_nc.is_contiguous()
    Kc = K.clone().requires_grad_(True)
    pl = pv.detach().requires_grad_(True)                                   # a leaf on the misaligned storage
    ff.utils.math.transform_points(pl, Kc).backward(g_nc)
    d_ref, dT_ref = full_bwd(ff, torch.from_numpy(p).cuda(), K, torch.from_numpy(g).cuda(), False)
    assert torch.equal(Kc.grad, dT_ref)
    assert torch.equal(pl.grad, d_ref)
    ref, scale = closed_form(p, K.cpu().numpy(), g, False)
    within(Kc.grad.cpu().numpy(), ref, scale, 1e-5)


# ---- the projector texture and the epipolar lines ------------------------------------------------------------------------
_A01 = torch.tensor([[0.5, 0.0, 0.0, 0.5], [0.0, 0.5, 0.0, 0.5], [0.0, 0.0, 1.0, 0.0], [0.0, 0.0, 0.0, 1.0]])
_FLIP = torch.diag(torch.tensor([1.0, -1.0, 1.0, 1.0]))
BLUR = ((5, 5), (3.0, 3.0))


def perspective01():
    return _A01 @ O.build_projection_matrix(60, 0.01, 1000.0)


def make_laser(ff, rays, K, device="cuda"):
    return ff.projection.Laser(ff.entity.Transformable("projector"), rays.to(device), K.to(device), 60.0, 0.01, 1000.0)


def oracle_texture(rays, K, sigma, ts, blur, points=None):
    if points is None:
        points = O.rays_to_ndc(rays, K)[:, 0:2]
    tex = O.reduce_sum(O.splat_dense(points, sigma, ts))
    if blur is not None:
        tex = O.gaussian_blur2d(tex, *blur)
    zero = torch.zeros_like(tex)
    return torch.stack([zero, tex, zero]).movedim(0, -1)


def oracle_k_grad(rays, K, sigma, ts, blur, w):
    """d (tex * w).sum() / d K by autograd of the oracle composition, and the per-entry error that ray-gradient errors within
    close_grad's 1e-4 budget can cause: the sum over rays of |d h_i| |p~_j|, with each ray's d ndc taken at
    max(||d ndc||, 0.1 mean ||d ndc||) in every component."""
    Kr = K.clone().requires_grad_(True)
    (oracle_texture(rays, Kr, sigma, ts, blur) * w).sum().backward()
    pts = O.rays_to_ndc(rays, K)[:, 0:2].detach().requires_grad_(True)
    (oracle_texture(rays, K, sigma, ts, blur, points=pts) * w).sum().backward()
    nrm = pts.grad.double().norm(dim=1)
    a = torch.maximum(nrm, 0.1 * nrm.mean())                                 # bound on each |d ndc| component
    pt = torch.cat([rays.double(), torch.ones(rays.shape[0], 1, dtype=torch.float64)], 1)
    h = pt @ (K.double() @ _FLIP.double()).T
    w3 = h[:, 3].abs()
    dh = torch.stack([a / w3, a / w3, torch.zeros_like(a), a * (h[:, 0].abs() + h[:, 1].abs()) / (w3 * w3)], 1)
    return Kr.grad, dh.T @ pt.abs()                                          # |d_M F| = |d_M| entry by entry


@pytest.mark.parametrize("ts,blur", [([128, 96], BLUR), ([96, 96], BLUR), ([128, 96], None), ([96, 96], None)])
def test_projector_texture_perspective_gradient(ff, ts, blur):
    rays = O.uniform_rays(0.06, 8, 8)
    K = perspective01()
    w = torch.randn((ts[1], ts[0], 3), generator=torch.Generator().manual_seed(14))
    laser = make_laser(ff, rays, K)
    laser._perspective.requires_grad_(True)
    laser._rays.requires_grad_(True)
    (laser.projector_texture(10.0, ts, blur=blur) * w.cuda()).sum().backward()
    ref, scale = oracle_k_grad(rays, K, 10.0, ts, blur, w)
    within(laser._perspective.grad.cpu().numpy(), ref.numpy(), scale.numpy() + ref.abs().numpy(), 1e-4)
    rr = rays.clone().requires_grad_(True)
    (oracle_texture(rr, K, 10.0, ts, blur) * w).sum().backward()
    close_grad(laser._rays.grad, rr.grad)


def test_epipolar_lines_camera_pose_gradient(ff):
    Laser = ff.projection.Laser
    rays = Laser.generate_uniform_rays(0.02, 4, 4)
    K = ff.utils.io.build_projection_matrix(60, 0.01, 1000.0)
    laser = Laser(ff.entity.Transformable("projector"), rays, K, 60.0, 0.5, 5.0)
    c, s = np.cos(0.1), np.sin(0.1)
    cam0 = torch.tensor([[c, 0, s, 0.3], [0, 1, 0, -0.1], [-s, 0, c, 0.2], [0, 0, 0, 1]], dtype=torch.float32)
    w = torch.randn((16, 48, 64), generator=torch.Generator().manual_seed(15))
    cam = cam0.cuda().requires_grad_(True)
    (laser.render_epipolar_lines(6.0, torch.tensor([64, 48]), camera_to_world=cam) * w.cuda()).sum().backward()
    lo = (laser.originPerRay() + 0.5 * laser.rays()).detach().cpu()
    hi = (laser.originPerRay() + 5.0 * laser.rays()).detach().cpu()
    Kc = (K.cpu() if torch.is_tensor(K) else torch.as_tensor(K)).float()
    camr = cam0.clone().requires_grad_(True)
    w2c = camr.inverse()
    lo2 = O.transform_points(O.transform_points(lo, w2c), Kc)[:, 0:2]
    hi2 = O.transform_points(O.transform_points(hi, w2c), Kc)[:, 0:2]
    (O.rasterize_lines(torch.stack([lo2, hi2], dim=1), 6.0, [64, 48]) * w).sum().backward()
    ref = camr.grad
    close(cam.grad, ref, rtol=1e-4, atol=1e-4 * float(ref.abs().max()))


# ---- TextureStep ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ts,blur,dtype", [([128, 96], BLUR, torch.float32), ([96, 96], None, torch.float32),
                                           ([128, 96], BLUR, torch.float64)])
def test_texture_step_perspective_gradient(ff, ts, blur, dtype):
    rays = O.uniform_rays(0.06, 8, 8)
    K = perspective01().to(dtype)
    g = torch.randn((8, ts[1], ts[0], 3), generator=torch.Generator().manual_seed(16)).cuda()
    ref_laser = make_laser(ff, rays, K)
    ref_laser._perspective.requires_grad_(True)
    (ref_laser.projector_texture(10.0, ts, blur=blur) * g.sum(0)).sum().backward()
    _, scale = oracle_k_grad(rays, K.float(), 10.0, ts, blur, g.sum(0).cpu())

    plain = ff.TextureStep(make_laser(ff, rays, K), sigma=10.0, texture_size=ts, blur=blur)
    plain.texture()
    d_plain = plain.backward(g).clone()
    assert plain.laser._perspective.grad is None

    laser = make_laser(ff, rays, K)
    laser._perspective.requires_grad_(True)
    laser._rays.requires_grad_(True)
    step = ff.TextureStep(laser, sigma=10.0, texture_size=ts, blur=blur)
    step.texture()
    d = step.backward(g).clone()
    gK = laser._perspective.grad.clone()
    assert gK.dtype == dtype and gK.shape == (4, 4)
    within(gK.cpu().numpy(), ref_laser._perspective.grad.cpu().numpy(), scale.numpy(), 1e-5)
    # the splat backward sums with float atomics, so two steps agree to rounding; from the same d ndc the fused pass writes the
    # points-only kernel's ray gradient bit for bit
    close_grad(d, d_plain, rtol=1e-5)
    rays_dev, M = step._saved[0], step._saved[1]
    assert torch.equal(d, points_bwd(ff, rays_dev, M, step._bufs["d_ndc"], False))
    assert torch.equal(laser._rays.grad, d)
    d2 = step.backward(g).clone()                          # a second call accumulates like autograd
    close_grad(d2, d, rtol=1e-5)
    assert torch.equal(laser._rays.grad, d + d2)
    within(laser._perspective.grad.cpu().numpy(), 2 * gK.cpu().numpy(), scale.numpy(), 1e-5)


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
    singles = [dist.new_group([r]) for r in range(world)]
    ts, B = [128, 96], 8 * world
    rays, K = O.uniform_rays(0.06, 8, 8), perspective01()
    g = torch.randn((B, ts[1], ts[0], 3), generator=torch.Generator().manual_seed(17)).to(dev)
    _, scale = oracle_k_grad(rays, K, 10.0, ts, BLUR, g.sum(0).cpu())

    def laser():
        las = make_laser(ff, rays, K, dev)
        las._perspective.requires_grad_(True)
        return las
    sharded_laser = laser()
    sharded = ff.TextureStep(sharded_laser, sigma=10.0, texture_size=ts, blur=BLUR)
    sharded.texture()
    calls, real = [0], dist.all_reduce

    def counting(*a, **k):
        calls[0] += 1
        return real(*a, **k)
    dist.all_reduce = counting
    try:
        d = sharded.backward(g[rank::world]).clone()
    finally:
        dist.all_reduce = real
    assert calls[0] == 1, calls
    gK = sharded_laser._perspective.grad.clone()
    full_laser = laser()
    full = ff.TextureStep(full_laser, sigma=10.0, texture_size=ts, blur=BLUR, process_group=singles[rank])
    full.texture()
    ref = full.backward(g).clone()
    close_grad(d, ref, rtol=1e-5)
    within(gK.cpu().numpy(), full_laser._perspective.grad.cpu().numpy(), scale.numpy(), 1e-5)
    for x in (d, gK):
        gathered = [torch.empty_like(x) for _ in range(world)]
        dist.all_gather(gathered, x)
        assert all(torch.equal(y, gathered[0]) for y in gathered)
    torch.cuda.synchronize()


def test_texture_step_perspective_two_ranks(ff):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port()), nprocs=2, join=True)
