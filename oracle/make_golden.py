"""TEST INFRASTRUCTURE ONLY -- writes ``tests/golden/*.npz`` by running the REAL reference
(a checkout of the original Fireflies project, imported through ``oracle/ref_loader.py``) on CPU.

Run with the reference at hand:  ``FIREFLIES_REF=<checkout> python oracle/make_golden.py``.
The fixtures pin ``oracle/ff_oracle.py`` (and, on the GPU box, the CUDA path) to outputs of
the reference's own code, because the reference ships no tests or golden vectors of its own.
"""
import os
import random
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
CPU = torch.device("cpu")


def npy(t):
    return t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)


def splat_case(ff, name, points, sigma, ts, store_full=True, stride=1):
    """dense + all four baked variants + L1 / weighted-sum gradients from the reference."""
    R = ff.graphics.rasterization
    tsz = torch.tensor(ts)
    sig_t = torch.tensor([float(sigma)])
    out = {"points": npy(points), "sigma": np.float32(sigma), "texture_size": np.array(ts)}
    n, h, w = points.shape[0], ts[1], ts[0]
    if n * h * w <= 30_000_000:
        p = points.clone().requires_grad_(True)
        dense = R.rasterize_points(p, float(sigma), tsz, device=CPU)
        S, O = R.sum(dense), R.softor(dense)
        loss = torch.nn.L1Loss()(O, S)
        loss.backward()
        out.update(dense_sum=npy(S)[::stride, ::stride], dense_softor=npy(O)[::stride, ::stride],
                   dense_l1=npy(loss), dense_l1_grad=npy(p.grad))
        if store_full and n <= 4:
            out["dense"] = npy(dense)
        g = torch.Generator().manual_seed(7)
        wS, wO = torch.randn(h, w, generator=g), torch.randn(h, w, generator=g)
        if stride == 1:
            out.update(wS=npy(wS), wO=npy(wO))   # else: regenerate in the test with torch.Generator().manual_seed(7)
        p = points.clone().requires_grad_(True)
        dense = R.rasterize_points(p, float(sigma), tsz, device=CPU)
        ((R.sum(dense) * wS).sum() + (R.softor(dense) * wO).sum()).backward()
        out["dense_weighted_grad"] = npy(p.grad)
    else:
        g = torch.Generator().manual_seed(7)
        wS, wO = torch.randn(h, w, generator=g), torch.randn(h, w, generator=g)
    # baked variants (sigma must be a tensor for these)
    b1 = R.baked_sum(points, sig_t, tsz, device=CPU)
    b2 = R.baked_sum_2(points, sig_t, tsz, device=CPU)
    o1 = R.baked_softor(points, sig_t, tsz, device=CPU)
    o2 = R.baked_softor_2(points, sig_t, tsz, device=CPU)
    out.update(baked_sum=npy(b1)[::stride, ::stride], baked_sum_2=npy(b2)[::stride, ::stride],
               baked_softor=npy(o1)[::stride, ::stride], baked_softor_2=npy(o2)[::stride, ::stride],
               baked_sum_total=np.float64(npy(b1).astype(np.float64).sum()),
               baked_softor_total=np.float64(npy(o1).astype(np.float64).sum()))
    # the in-tree pattern-optimisation step (rasterization.py:589-600)
    p = points.clone().requires_grad_(True)
    summed = R.baked_sum_2(p, sig_t, tsz, device=CPU)
    softored = R.baked_softor_2(p, sig_t, tsz, device=CPU)
    loss = torch.nn.L1Loss()(softored, summed) if ts[0] == ts[1] else torch.nn.L1Loss()(softored, summed.T)
    loss.backward()
    out.update(baked_l1=npy(loss), baked_l1_grad=npy(p.grad))
    # weighted: <wS, baked_sum> + <wO, baked_softor_2>, weights in the dense orientation
    p = points.clone().requires_grad_(True)
    L = (R.baked_sum_2(p, sig_t, tsz, device=CPU).T * wS).sum() + (R.baked_softor_2(p, sig_t, tsz, device=CPU) * wO).sum()
    L.backward()
    out["baked_weighted_grad"] = npy(p.grad)
    out["stride"] = np.int64(stride)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print("wrote", name, {k: v.shape for k, v in out.items() if hasattr(v, "shape") and v.ndim})


def transform_cases(ff):
    Mesh = ff.entity.Mesh
    US = ff.sampling.UniformSampler
    out = {}
    # KAT2: fixed samplers
    verts = torch.tensor([[1.0, 2.0, 3.0], [-1.0, 0.5, 0.25]])
    m = Mesh("m", verts, device=CPU)
    m.set_centroid(torch.tensor([[0.5, -0.5, 2.0]]))
    m.set_rotation_sampler(US(torch.tensor([0.1, 0.2, 0.3]), torch.tensor([0.1, 0.2, 0.3]), device=CPU))
    m.set_translation_sampler(US(torch.tensor([1.0, 2.0, 3.0]), torch.tensor([1.0, 2.0, 3.0]), device=CPU))
    m.set_scale_sampler(US(torch.tensor([2.0, 1.0, 0.5]), torch.tensor([2.0, 1.0, 0.5]), device=CPU))
    m.set_randomizable(True)
    m.train()
    m.randomize()
    out.update(kat2_verts=npy(verts), kat2_world=npy(m.world()), kat2_out=npy(m.get_randomized_vertices()))

    # seeded random T/R/S with a non-identity world, 8 successive draws; u variates replayed
    g = torch.Generator().manual_seed(11)
    verts = torch.rand(257, 3, generator=g) * 2 - 1
    W0 = torch.eye(4)
    W0[:3, :3] = torch.tensor([[0.0, -1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 1.0]]) * 1.5
    W0[:3, 3] = torch.tensor([0.3, -0.2, 0.1])
    m = Mesh("r", verts, device=CPU)
    m.set_world(W0)
    m.set_centroid(torch.tensor([[0.25, 0.5, -0.75]]))
    m.rotate(torch.tensor([-0.5, -1.0, -3.0]), torch.tensor([0.5, 1.0, 3.0]))
    m.translate(torch.tensor([-1.0, -2.0, -3.0]), torch.tensor([1.0, 2.0, 3.0]))
    m.scale(torch.tensor([0.5, 0.8, 1.0]), torch.tensor([2.0, 1.2, 3.0]))
    m.train()
    torch.manual_seed(1234)
    worlds, outs = [], []
    for _ in range(8):
        m.randomize()
        worlds.append(npy(m.world()))
        outs.append(npy(m.get_randomized_vertices()))
    torch.manual_seed(1234)
    u = torch.stack([torch.rand(3) for _ in range(8 * 3)]).view(8, 3, 3)   # draw order T, R, S (SURVEY KAT5)
    out.update(rand_verts=npy(verts), rand_world0=npy(W0), rand_centroid=np.array([0.25, 0.5, -0.75], np.float32),
               rand_min=np.array([[-1, -2, -3], [-0.5, -1, -3], [0.5, 0.8, 1.0]], np.float32),
               rand_max=np.array([[1, 2, 3], [0.5, 1, 3], [2.0, 1.2, 3.0]], np.float32),
               rand_u=npy(u), rand_worlds=np.stack(worlds), rand_outs=np.stack(outs))

    # parent -> child chain (examples/03_parent_child.py), rotate_z on the parent, eval mode
    g = torch.Generator().manual_seed(12)
    va, vb = torch.rand(33, 3, generator=g), torch.rand(17, 3, generator=g)
    a, b = Mesh("a", va, device=CPU), Mesh("b", vb, device=CPU)
    a.set_centroid(torch.tensor([[1.0, 0.0, 0.0]]))
    b.set_centroid(torch.tensor([[0.0, 2.0, 0.0]]))
    b.setParent(a)
    b.set_randomizable(True)
    a.rotate_z(-np.pi, np.pi)
    a.eval(); b.eval()
    cw, cv, rot = [], [], []
    for _ in range(5):
        a.randomize(); b.randomize()
        rot.append(npy(a._sampled_rotation).copy())
        cw.append(np.stack([npy(a.world()), npy(b.world())]))
        cv.append(npy(b.get_randomized_vertices()))
    out.update(chain_va=npy(va), chain_vb=npy(vb), chain_rot=np.stack(rot), chain_worlds=np.stack(cw),
               chain_child_verts=np.stack(cv))

    # non-mesh Transformable (no scale) + attribute draws (entity/base.py:220-234)
    t = ff.entity.Transformable("light", device=CPU)
    t.set_world(W0.clone())
    t.rotate_x(-0.3, 0.3)
    t.translate_y(-1.0, 1.0)
    t.add_float_key("power", 1.0, 3.0)
    t.add_vec3_key("color", torch.tensor([0.0, 0.1, 0.2]), torch.tensor([1.0, 0.9, 0.8]))
    t.add_vec3_sampler("intensity", ff.sampling.UniformScalarToVec3Sampler(0.1, 10.0, device=CPU))
    t.train()
    torch.manual_seed(99)
    tw, tf, tv, ti = [], [], [], []
    for _ in range(4):
        t.randomize()
        tw.append(npy(t.world()))
        tf.append(npy(t.get_randomized_float_attributes()["power"]).copy())
        tv.append(npy(t.get_randomized_vec3_attributes()["color"]).copy())
        ti.append(npy(t.get_randomized_vec3_attributes()["intensity"]).copy())
    torch.manual_seed(99)
    us = []
    for _ in range(4):   # draw order: translation(3), rotation(3), power(1), color(3), intensity(1)
        us.append(np.concatenate([npy(torch.rand(3)), npy(torch.rand(3)), npy(torch.rand(1)), npy(torch.rand(3)), npy(torch.rand(1))]))
    out.update(tr_world0=npy(W0), tr_worlds=np.stack(tw), tr_power=np.stack(tf), tr_color=np.stack(tv),
               tr_intensity=np.stack(ti), tr_u=np.stack(us))

    # transform_points / transform_directions with a projective matrix
    g = torch.Generator().manual_seed(13)
    pts = torch.rand(101, 3, generator=g) * 4 - 2
    K = ff.utils.io.build_projection_matrix(60, 0.01, 1000.0, device=CPU) if hasattr(ff.utils, "io") else None
    if K is None:
        import fireflies.utils.io as io
        K = io.build_projection_matrix(60, 0.01, 1000.0, device=CPU)
    out.update(tp_pts=npy(pts), tp_K=npy(K), tp_out=npy(ff.utils.math.transform_points(pts, K)),
               td_out=npy(ff.utils.math.transform_directions(pts, W0)))
    np.savez_compressed(os.path.join(OUT, "transforms.npz"), **out)
    print("wrote transforms")


def sampler_cases(ff):
    S = ff.sampling
    out = {}
    # KAT4: eval stepping with aliasing
    us = S.UniformSampler(torch.zeros(3), torch.zeros(3), device=CPU)
    us.get_min()[2], us.get_max()[2] = -np.pi, np.pi     # what rotate_z(-pi, pi) does
    us.eval()
    out["eval_vec3"] = np.stack([npy(us.sample()).copy() for _ in range(12)])
    sc = S.UniformSampler(0.0, 0.05, device=CPU)
    sc.eval()
    out["eval_scalar"] = np.stack([npy(sc.sample()).copy() for _ in range(14)])
    v3 = S.UniformSampler(torch.tensor([0.0, 1.0, -1.0]), torch.tensor([0.035, 1.5, 0.0]), device=CPU)
    v3.eval()
    out["eval_vec3_ranged"] = np.stack([npy(v3.sample()).copy() for _ in range(12)])
    s2v = S.UniformScalarToVec3Sampler(0.1, 10.0, device=CPU)
    s2v.eval()
    out["eval_s2v"] = np.stack([npy(s2v.sample()).copy() for _ in range(4)])
    an = S.AnimationSampler(0, 5, 0, 5, device=CPU)
    an.eval()
    out["anim_eval"] = np.array([an.sample() for _ in range(9)], np.int64)
    an.train()
    random.seed(1)
    out["anim_train_seed1"] = np.array([an.sample() for _ in range(5)], np.int64)
    # train-mode uniform draws with their u variates
    tr = S.UniformSampler(torch.tensor([-1.0, 0.0, 2.0]), torch.tensor([1.0, 0.5, 2.0]), device=CPU)
    torch.manual_seed(5)
    out["train_uniform"] = np.stack([npy(tr.sample()) for _ in range(6)])
    torch.manual_seed(5)
    out["train_uniform_u"] = np.stack([npy(torch.rand(3)) for _ in range(6)])
    np.savez_compressed(os.path.join(OUT, "samplers.npz"), **out)
    print("wrote samplers")


def fireflies_transform(ff, pts, T):
    return sys.modules["fireflies.utils.math"].transform_points(pts, T)


def laser_cases(ff):
    import fireflies.utils.io as io
    Laser = ff.projection.Laser
    out = {}
    rays = Laser.generate_uniform_rays(0.0275, 18, 18, device=CPU)
    K = io.build_projection_matrix(60, 0.01, 1000.0, device=CPU)
    tr = ff.entity.Transformable("projector", device=CPU)
    laser = Laser(tr, rays, K, 60.0, 0.01, 1000.0, device=CPU)
    ndc = laser.projectRaysToNDC()
    back = laser.projectNDCPointsToWorld(ndc.clone())
    out.update(rays=npy(rays), K=npy(K), ndc=npy(ndc), back=npy(back))
    # clamp_to_fov expects NDC in [0,1]: use a K that maps there (0.5*x+0.5)
    A = torch.tensor([[0.5, 0, 0, 0.5], [0, 0.5, 0, 0.5], [0, 0, 1.0, 0], [0, 0, 0, 1.0]])
    K01 = A @ K
    wide = Laser.generate_uniform_rays(0.09, 9, 9, device=CPU)
    laser2 = Laser(tr, wide.clone(), K01, 60.0, 0.01, 1000.0, device=CPU)
    ndc2 = laser2.projectRaysToNDC()
    laser2.clamp_to_fov()
    out.update(K01=npy(K01), wide=npy(wide), wide_ndc=npy(ndc2), wide_clamped=npy(laser2._rays))
    tex = laser.generateTexture(10.0, torch.tensor([64, 48]))
    pts01 = (ndc[:, 0:2] * 0.5 + 0.5)
    out.update(gen_tex_sum=npy(tex.sum(0)), pts01=npy(pts01))
    # out-of-bounds respawn (laser.py:208-249): the reference draws torch.rand(K, 3) for its K out-of-bounds rays
    wider = Laser.generate_uniform_rays(0.17, 9, 9, device=CPU)
    laser3 = Laser(tr, wider.clone(), K01, 60.0, 0.01, 1000.0, device=CPU)
    xy = fireflies_transform(ff, wider, K01)[:, 0:2]
    K_oob = int(((xy >= 1.0) | (xy <= 0.0)).any(dim=1).sum())
    torch.manual_seed(11)
    var = torch.rand(K_oob, 3)
    torch.manual_seed(11)
    laser3.randomize_laser_out_of_bounds()
    out.update(respawn_rays=npy(wider), respawn_variates=npy(var), respawn_laser=npy(laser3._rays), respawn_k=np.int32(K_oob))
    laser4 = Laser(tr, wide.clone(), K01, 60.0, 0.01, 1000.0, device=CPU)
    cam_ndc = ndc2.clone()
    cam_ndc[:, 0:2] = cam_ndc[:, 0:2] * 2.0 - 0.6
    xy = cam_ndc[:, 0:2]
    K_cam = int(((xy >= 1.0) | (xy <= -1.0)).any(dim=1).sum())
    torch.manual_seed(12)
    var2 = torch.rand(K_cam, 3)
    torch.manual_seed(12)
    laser4.randomize_camera_out_of_bounds(cam_ndc)
    out.update(respawn_cam_ndc=npy(cam_ndc), respawn_cam_variates=npy(var2), respawn_cam=npy(laser4._rays), respawn_cam_k=np.int32(K_cam))
    inside = Laser.generate_uniform_rays(0.01, 5, 5, device=CPU)       # nothing out of bounds: rays must stay untouched (not renormalised)
    inside = inside * 1.5
    laser5 = Laser(tr, inside.clone(), K01, 60.0, 0.01, 1000.0, device=CPU)
    laser5.randomize_laser_out_of_bounds()
    out.update(respawn_inside=npy(inside), respawn_inside_after=npy(laser5._rays))
    # generate_uniform_rays_by_count (laser.py:40-66): deterministic
    out["by_count_5x4"] = npy(Laser.generate_uniform_rays_by_count(5, 4, K01, device=CPU))
    out["by_count_3x3_K"] = npy(Laser.generate_uniform_rays_by_count(3, 3, K, device=CPU))
    np.savez_compressed(os.path.join(OUT, "laser.npz"), **out)
    print("wrote laser")


def post_cases(ff):
    P = ff.postprocessing
    out = {}
    g = np.random.default_rng(3)
    img = g.random((37, 53), dtype=np.float32)
    wn = P.WhiteNoise(0.02, 0.05, 1.0)
    np.random.seed(21)
    res = wn.post_process(img.copy())
    np.random.seed(21)
    noise = np.random.normal(np.ones_like(img) * 0.02, np.ones_like(img) * 0.05)
    out.update(img=img, wn_out=res, wn_noise=noise)
    # gates: random.uniform(0,1) < p per function, chain order (postprocessing/base.py:10-14)
    random.seed(6)
    calls = []

    class Probe(P.BasePostProcessingFunction):
        def __init__(self, p, tag):
            super().__init__(p)
            self.tag = tag

        def post_process(self, image):
            calls.append(self.tag)
            return image

    pp = P.PostProcessor([Probe(0.5, 0), Probe(0.5, 1)])
    gates = []
    for _ in range(16):
        calls.clear()
        pp.post_process(img)
        gates.append([0 in calls, 1 in calls])
    out["gates_seed6"] = np.array(gates)
    # ApplySilhouette (postprocessing/apply_silhouette.py:17-40) run as the reference runs it: its own random.randint draws and the
    # REAL cv2.circle (OpenCV is installed; only kornia is not, so kornia.filters.gaussian_blur2d is the restated blur).  A frame of
    # ones makes the result the blurred disc itself, which is what pins the rasterisation of the disc.
    from oracle import ff_oracle as O
    sys.modules["kornia.filters"].gaussian_blur2d = lambda x, k, sg: O.gaussian_blur2d(x, k, tuple(float(v) for v in sg))
    sys.modules["kornia"].filters = sys.modules["kornia.filters"]
    sil = P.ApplySilhouette()
    ones = np.ones((512, 448), dtype=np.float32)
    grad = (np.add.outer(np.arange(512), np.arange(448)) / 960.0).astype(np.float32)
    discs, outs = [], []
    for seed, frame in ((4, ones), (5, ones), (6, grad)):
        random.seed(seed)
        cx, cy, r = random.randint(100, 200), random.randint(200, 300), random.randint(170, 230)
        random.seed(seed)
        outs.append(np.asarray(sil.post_process(frame.copy()), dtype=np.float32))
        discs.append([cx, cy, r])
    out.update(silhouette_discs=np.array(discs, dtype=np.int32), silhouette_seeds=np.array([4, 5, 6]), silhouette_out=np.stack(outs),
               silhouette_grad=grad)
    np.savez_compressed(os.path.join(OUT, "postprocess.npz"), **out)
    print("wrote postprocess")


def line_depth_cases(ff):
    """rasterize_lines (+ L1(softor, sum) gradient, test_line_reg rasterization.py:684-697), rasterize_depth,
    subsampled_point_raster from the reference.  The reference scales `lines` in place (:122-123): it gets clones."""
    R = ff.graphics.rasterization
    out = {}
    # KAT3 (SURVEY App. B)
    kat = torch.tensor([[[0.2, 0.2], [0.8, 0.6]]])
    out["kat3_lines"] = npy(kat)
    out["kat3"] = npy(R.rasterize_lines(kat.clone(), torch.tensor([4.0]), torch.tensor([8, 6]), device=CPU))
    g = torch.Generator().manual_seed(5)
    lines = torch.rand(12, 2, 2, generator=g) * 1.2 - 0.1           # some end points outside [0,1]
    lines[3, 1] = lines[3, 0]                                       # degenerate segment: the eps guard (:142)
    ts = [96, 64]
    out["lines"], out["lines_ts"], out["lines_sigma"] = npy(lines), np.array(ts), np.float32(10.0)
    l = lines.clone().requires_grad_(True)
    tex = R.rasterize_lines(l * 1.0, torch.tensor([10.0]), torch.tensor(ts), device=CPU)
    out["lines_dense"] = npy(tex)
    S, O = tex.sum(dim=0), R.softor(tex)
    out["lines_sum"], out["lines_softor"] = npy(S), npy(O)
    loss = torch.nn.L1Loss()(O, S)
    loss.backward()
    out["lines_l1"], out["lines_l1_grad"] = npy(loss), npy(l.grad)
    gw = torch.Generator().manual_seed(6)
    wS, wO = torch.randn(ts[1], ts[0], generator=gw), torch.randn(ts[1], ts[0], generator=gw)
    l = lines.clone().requires_grad_(True)
    tex = R.rasterize_lines(l * 1.0, torch.tensor([10.0]), torch.tensor(ts), device=CPU)
    ((tex.sum(dim=0) * wS).sum() + (R.softor(tex) * wO).sum()).backward()
    out["lines_wS"], out["lines_wO"], out["lines_weighted_grad"] = npy(wS), npy(wO), npy(l.grad)
    # depth
    pts = torch.rand(9, 3, generator=g)
    pts[0, 0:2] = torch.tensor([1.05, 0.5])                         # outside the frame: the maximum sits on the border
    out["depth_points"], out["depth_ts"], out["depth_sigma"] = npy(pts), np.array([40, 24]), np.float32(6.0)
    out["depth_dense"] = npy(R.rasterize_depth(pts[:, 0:2], pts[:, 2:3], 6.0, torch.tensor([40, 24]), device=CPU))
    sub = R.subsampled_point_raster.__wrapped__ if hasattr(R.subsampled_point_raster, "__wrapped__") else None
    # subsampled_point_raster calls rasterize_depth with the default device (cuda): restate its four lines on CPU
    levels = []
    for i in range(3):
        d = R.rasterize_depth(pts[:, 0:2], pts[:, 2:3], 6.0, torch.tensor([40, 24]) // 2 ** i, device=CPU)
        levels.append(npy(R.softor(d, keepdim=True)))
    for i, lv in enumerate(levels):
        out[f"depth_level{i}"] = lv
    # rasterize_points_in_non_ndc (rasterization.py:38-63): points in texel units
    ppx = torch.tensor([[3.25, 7.5], [20.0, 11.0], [-2.0, 5.0], [39.5, 23.75]])
    lp = ppx.clone().requires_grad_(True)
    tex = R.rasterize_points_in_non_ndc(lp, 6.0, torch.tensor([40, 24]), device=CPU)
    gw2 = torch.randn(4, 24, 40, generator=torch.Generator().manual_seed(8))
    (tex * gw2).sum().backward()
    out.update(px_points=npy(ppx), px_dense=npy(tex), px_w=npy(gw2), px_grad=npy(lp.grad))
    np.savez_compressed(os.path.join(OUT, "lines_depth.npz"), **out)


def perlin_cases(ff):
    """rand_perlin_2d_octaves and NoiseTextureLerpSampler.sample_train from the reference under a fixed seed, plus the
    torch.rand lattice draws it consumed (re-drawn under the same seed)."""
    import fireflies.sampling.noise_texture_lerp as NT
    out = {}
    for name, shape, res, octaves, pers, seed in [("a", [64, 64], (2, 2), 3, 0.5, 21), ("b", [96, 128], (4, 8), 2, 1.7, 22),
                                                   ("c", [128, 128], (8, 8), 4, 0.3, 23)]:
        torch.manual_seed(seed)
        noise = NT.rand_perlin_2d_octaves(shape, res, octaves, pers)
        torch.manual_seed(seed)
        angles, f = [], 1
        for _ in range(octaves):
            angles.append(torch.rand(f * res[0] + 1, f * res[1] + 1)); f *= 2
        out[f"{name}_noise"] = npy(noise)
        out[f"{name}_cfg"] = np.array([shape[0], shape[1], res[0], res[1], octaves], dtype=np.int64)
        out[f"{name}_pers"] = np.float64(pers)
        out[f"{name}_angles"] = npy(torch.cat([a.reshape(-1) for a in angles]))
    # the whole sampler: python `random` for (i, octaves, persistence), torch.rand for the lattice
    ca, cb = torch.tensor([0.8, 0.14, 0.34]), torch.tensor([0.1, 0.4, 0.9])
    smp = NT.NoiseTextureLerpSampler(ca, cb, [128, 128], device=CPU)
    random.seed(31); torch.manual_seed(31)
    tex = smp.sample_train()
    out.update(sampler_tex=npy(tex), sampler_ca=npy(ca), sampler_cb=npy(cb))
    np.savez_compressed(os.path.join(OUT, "perlin.npz"), **out)
    print("wrote perlin")


class _OracleCurve:
    """Stand-in for geomdl's NURBS.Curve (absent here): the attributes utils/io.py:105-108 sets, evaluated by the oracle's
    restatement.  What the fixtures pin is the reference's Curve arithmetic AROUND the evaluator."""
    def __init__(self, degree, ctrlpts, knotvector, weights=None):
        from oracle import ff_oracle as O
        self.degree, self.ctrlpts, self.weights = degree, ctrlpts, weights
        self.knotvector = O.nurbs_normalize_knots(knotvector)
        self._O = O

    def evaluate_single(self, t):
        return self._O.nurbs_curve_point(self.ctrlpts, self.knotvector, self.degree, t, self.weights)


CURVE_CTRL = [[0.0, 0.0, 0.0], [1.0, 2.0, 0.5], [3.0, 2.5, -1.0], [4.0, 0.0, 2.0], [6.0, -1.0, 1.0], [7.5, 0.5, 0.0], [9.0, 2.0, 3.0]]
CURVE_KNOTS = [0.0, 0.0, 0.0, 0.0, 1.0, 2.0, 2.5, 4.0, 4.0, 4.0, 4.0]
CURVE_WEIGHTS = [1.0, 0.7, 1.3, 1.0, 2.0, 0.5, 1.0]


def curve_cases(ff):
    """The reference's Curve (entity/curve.py) driven through train / eval randomize() with the oracle evaluator as its
    `_curve`.  Its constructor raises (`super().__init__(self, name, device)`, :24): the instance is assembled by hand
    with the constructor's own attribute values (:26-34)."""
    import random as pyrandom
    from fireflies.entity.curve import Curve
    from fireflies.entity.base import Transformable
    out = {}
    for tag, weights in (("bspline", None), ("rational", CURVE_WEIGHTS)):
        c = object.__new__(Curve)
        Transformable.__init__(c, "path", CPU)
        c._curve = _OracleCurve(3, CURVE_CTRL, CURVE_KNOTS, weights)
        c.curve_epsilon = 0.05; c.curve_delta = c.curve_epsilon
        c._interp_steps = 1000; c._interp_delta = 1.0 / c._interp_steps
        c.eval_interval_start = 0.05
        g = torch.Generator().manual_seed(41)
        W = torch.eye(4); W[0:3, 0:3] = torch.linalg.qr(torch.randn(3, 3, generator=g))[0]; W[0:3, 3] = torch.tensor([0.3, -1.0, 2.0])
        c.set_world(W)
        c.train(); pyrandom.seed(5)
        deltas, worlds = [], []
        for _ in range(3):
            c.randomize(); deltas.append(c.curve_delta); worlds.append(npy(c.world()))
        c.eval()
        for _ in range(40):
            c.randomize(); deltas.append(c.curve_delta); worlds.append(npy(c.world()))
        c.curve_delta = 0.9485      # walk over the wrap at 1 - epsilon (:88-89)
        for _ in range(4):
            c.randomize(); deltas.append(c.curve_delta); worlds.append(npy(c.world()))
        for t in (0.2, 0.5, 0.77):
            c.curve_delta = t
            out[f"{tag}_rot_{t}"] = npy(c.sample_rotation()); out[f"{tag}_trans_{t}"] = npy(c.sample_translation())
        out[f"{tag}_deltas"] = np.array(deltas, dtype=np.float64)
        out[f"{tag}_worlds"] = np.stack(worlds)
        out[f"{tag}_W"] = npy(W)
        ts = np.linspace(0.0, 1.0, 101)
        out[f"{tag}_points64"] = np.array([c._curve.evaluate_single(float(t)) for t in ts])
    out["ctrl"], out["knots"], out["weights"] = np.array(CURVE_CTRL), np.array(CURVE_KNOTS), np.array(CURVE_WEIGHTS)
    np.savez_compressed(os.path.join(OUT, "curve.npz"), **out)
    print("wrote curve")


def poisson_cases(ff):
    """bridson (sampling/poisson.py) under np.random.seed, Laser.generate_blue_noise_rays (laser.py:94-145),
    utils/intersections.py and rotation_matrix_from_vectors[_with_fixed_up] (utils/math.py:67-159) from the reference."""
    import fireflies.sampling.poisson as PS
    import fireflies.utils.intersections as IS
    out = {}
    np.random.seed(17)
    n, pts = PS.bridson(np.ones([48, 64]) * 5.5)
    out["uniform_pts"], out["uniform_n"] = pts, np.int64(n)
    rad = np.ones([40, 40]) * 6.0
    rad[10:30, 10:30] = 2.5
    np.random.seed(18)
    n, pts = PS.bridson(rad, k=12)
    out["varying_radius"], out["varying_pts"] = rad, pts
    import fireflies.utils.io as IO
    K = IO.build_projection_matrix(60.0, 0.01, 1000.0, device=CPU)
    np.random.seed(19)
    rays = ff.projection.Laser.generate_blue_noise_rays(64, 48, 60, K, device=CPU)
    out["blue_K"], out["blue_rays"] = npy(K), npy(rays)
    g = torch.Generator().manual_seed(51)
    o, d = torch.randn(33, 3, generator=g), torch.nn.functional.normalize(torch.randn(33, 3, generator=g), dim=1)
    po, pn = torch.randn(33, 3, generator=g), torch.nn.functional.normalize(torch.randn(33, 3, generator=g), dim=1)
    d[4] = torch.linalg.cross(pn[4], torch.tensor([0.3, 0.2, 0.9]))          # (nearly) parallel to the plane
    out.update(rp_o=npy(o), rp_d=npy(d), rp_po=npy(po), rp_pn=npy(pn), rp_t=npy(IS.rayPlane(o, d, po, pn)))
    a, b = torch.rand(50, 2, generator=g) * 10, torch.rand(50, 2, generator=g) * 10
    ra, rb = torch.rand(50, 1, generator=g) * 2, torch.rand(50, 1, generator=g) * 2
    out.update(ss_a=npy(a), ss_b=npy(b), ss_ra=npy(ra), ss_rb=npy(rb), ss_hit=IS.sphereSphere(a, ra, b, rb).numpy())
    M = ff.utils.math
    v1, v2 = torch.tensor([0.0, 1.0, 0.0]), torch.tensor([0.3, -0.2, 0.8])
    out.update(rot_v1=npy(v1), rot_v2=npy(v2), rot=npy(M.rotation_matrix_from_vectors(v1, v2)),
               rot_up=npy(M.rotation_matrix_from_vectors_with_fixed_up(v1, v2)))
    np.savez_compressed(os.path.join(OUT, "poisson_misc.npz"), **out)
    print("wrote poisson_misc")


LIVE_CASES = [(7, [33, 21], 6.0), (40, [96, 64], 20.0), (5, [16, 16], 49.0)]      # (points, texture size, sigma)
LIVE_ANGLES = [0.0, 0.3, -2.5, 3.14159]


def live_reference_outputs(ff):
    """The reference's outputs that tests/test_oracle_golden.py::test_oracle_equals_live_reference compares the oracle with:
    dense / baked / full-frame rasterisation on seeded points (texture sizes of one odd, one large and one square case) and the
    yaw / pitch / roll matrices (the reference always receives an fp32 0-d tensor)."""
    R, m = ff.graphics.rasterization, ff.utils.math
    gen = torch.Generator().manual_seed(123)
    out = {}
    for i, (n, ts, sigma) in enumerate(LIVE_CASES):
        pts = torch.rand(n, 2, generator=gen)
        tsz, sg, c = torch.tensor(ts), torch.tensor([sigma]), f"c{i}_"
        out.update({c + "points": npy(pts), c + "dense": npy(R.rasterize_points(pts, sigma, tsz, device=CPU)),
                    c + "baked_sum": npy(R.baked_sum(pts, sg, tsz, device=CPU)),
                    c + "baked_sum_2": npy(R.baked_sum_2(pts, sg, tsz, device=CPU)),
                    c + "baked_softor_2": npy(R.baked_softor_2(pts, sg, tsz, device=CPU)),
                    c + "baked_sum_std3": npy(R.baked_sum(pts, sg, tsz, num_std=3, device=CPU))})
        if ts[0] == ts[1]:   # the loop-over-points full-frame variants only work on square textures
            out[c + "points_baked_sum"] = npy(R.rasterize_points_baked_sum(pts, sigma, tsz, device=CPU))
            out[c + "points_baked_softor"] = npy(R.rasterize_points_baked_softor(pts, sigma, tsz, device=CPU))
    a32 = [torch.tensor(a) for a in LIVE_ANGLES]
    for key, fn in (("yaw", m.getYawTransform), ("pitch", m.getPitchTransform), ("roll", m.getRollTransform)):
        out[key] = np.stack([npy(fn(a, CPU)) for a in a32])
    return out


def live_reference_cases(ff):
    out = live_reference_outputs(ff)
    out["c1_dense"], out["c1_dense_stride"] = out["c1_dense"][:, ::2, ::2], np.int64(2)    # every other texel of [40,64,96]: 1 MB -> 250 kB
    out["source"] = np.array("the original Fireflies code, run by oracle/make_golden.py::live_reference_cases")
    np.savez_compressed(os.path.join(OUT, "live_reference.npz"), **out)
    print("wrote live_reference")


def reference_api(ff):
    """Names and positional signatures of the reference package (oracle/ref_loader.py::api) for tests/test_abi_cpu.py."""
    import json
    out = {"source": "the original Fireflies tree, read by oracle/make_golden.py::reference_api",
           **ref_loader.api(os.path.join(ref_loader.REF_ROOT, "fireflies"))}
    with open(os.path.join(OUT, "reference_api.json"), "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print("wrote reference_api")


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    ff = ref_loader.load()
    if len(sys.argv) > 1:          # python oracle/make_golden.py curve_cases poisson_cases: only those fixture files
        for name in sys.argv[1:]:
            globals()[name](ff)
        return
    # KAT1 (SURVEY App. B): point 2 exactly on pixel (3,4) -> g == 1
    splat_case(ff, "splat_kat1", torch.tensor([[0.25, 0.75], [0.5, 0.5]]), 4.0, [8, 6])
    g = torch.Generator().manual_seed(0)
    pts = torch.rand(24, 2, generator=g)
    pts[0] = torch.tensor([0.004, 0.5]); pts[1] = torch.tensor([0.5, 0.996]); pts[2] = torch.tensor([0.999, 0.001])
    pts[3] = torch.tensor([0.5, 0.5])    # exactly on a pixel centre for even sizes
    splat_case(ff, "splat_small_rect", pts, 9.0, [48, 40])
    g = torch.Generator().manual_seed(1)
    splat_case(ff, "splat_mid", torch.rand(64, 2, generator=g) * 0.96 + 0.02, 30.0, [128, 128])
    g = torch.Generator().manual_seed(0)
    splat_case(ff, "splat_c1", torch.rand(100, 2, generator=g) * 0.8 + 0.1, 100.0, [512, 512], stride=8)
    transform_cases(ff)
    sampler_cases(ff)
    laser_cases(ff)
    post_cases(ff)
    line_depth_cases(ff)
    perlin_cases(ff)
    curve_cases(ff)
    poisson_cases(ff)
    live_reference_cases(ff)
    reference_api(ff)


if __name__ == "__main__":
    main()
