"""CPU: pins ``oracle/ff_oracle.py`` to fixtures generated from the real reference
(``oracle/make_golden.py``), and also to the live reference when ``FIREFLIES_REF`` names a checkout of it."""
import random

import numpy as np
import pytest
import torch

from oracle import ff_oracle as O
from oracle import ref_loader

SPLAT_CASES = ["splat_kat1", "splat_small_rect", "splat_mid", "splat_c1"]


def T(a):
    return torch.from_numpy(np.asarray(a))


def close(a, b, rtol=1e-5, atol=1e-7):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    err = np.abs(a - b) - (atol + rtol * np.abs(b))
    assert err.max() <= 0, f"max violation {err.max():.3e}, max abs diff {np.abs(a - b).max():.3e}"


@pytest.mark.parametrize("case", SPLAT_CASES)
def test_splat_forward_matches_reference_fixture(golden, case):
    g = golden(case)
    pts, sigma, ts, st = T(g["points"]), float(g["sigma"]), g["texture_size"].tolist(), int(g["stride"])
    if "dense_sum" in g:
        dense = O.splat_dense(pts, sigma, ts)
        close(O.reduce_sum(dense)[::st, ::st], g["dense_sum"], atol=1e-6)
        close(O.softor(dense)[::st, ::st], g["dense_softor"], atol=1e-6)
        if "dense" in g:
            assert np.array_equal(dense.numpy(), g["dense"])          # same elementwise arithmetic -> bit-equal
    close(O.baked_sum(pts, sigma, ts)[::st, ::st], g["baked_sum"], atol=1e-6)
    close(O.baked_sum(pts, sigma, ts, transposed=True)[::st, ::st], g["baked_sum_2"], atol=1e-6)
    close(O.baked_softor(pts, sigma, ts)[::st, ::st], g["baked_softor"], atol=1e-6)
    close(O.baked_softor(pts, sigma, ts)[::st, ::st], g["baked_softor_2"], atol=1e-6)
    close(O.baked_sum(pts, sigma, ts).double().sum(), g["baked_sum_total"], rtol=1e-6)
    close(O.baked_softor(pts, sigma, ts).double().sum(), g["baked_softor_total"], rtol=1e-6)


@pytest.mark.parametrize("case", ["splat_kat1", "splat_small_rect", "splat_mid"])
def test_sequential_equals_scatter(golden, case):
    g = golden(case)
    pts, sigma, ts = T(g["points"]), float(g["sigma"]), g["texture_size"].tolist()
    close(O.baked_sum_sequential(pts, sigma, ts), O.baked_sum(pts, sigma, ts), atol=1e-6)
    close(O.baked_softor_sequential(pts, sigma, ts), O.baked_softor(pts, sigma, ts), atol=1e-6)


@pytest.mark.parametrize("case", SPLAT_CASES)
def test_splat_gradients_match_reference_fixture(golden, case):
    g = golden(case)
    pts, sigma, ts = T(g["points"]), float(g["sigma"]), g["texture_size"].tolist()
    h, w = ts[1], ts[0]
    if "wS" in g:
        wS, wO = T(g["wS"]), T(g["wO"])
    else:
        gen = torch.Generator().manual_seed(7)
        wS, wO = torch.randn(h, w, generator=gen), torch.randn(h, w, generator=gen)
    scale = np.abs(g["baked_weighted_grad"]).max()
    # autograd through the oracle's baked forms
    p = pts.clone().requires_grad_(True)
    ((O.baked_sum(p, sigma, ts) * wS).sum() + (O.baked_softor(p, sigma, ts) * wO).sum()).backward()
    close(p.grad, g["baked_weighted_grad"], rtol=1e-4, atol=1e-4 * scale)
    # closed-form fp64 gradient (what the CUDA backward implements)
    ana = O.splat_grad_analytic(pts, sigma, ts, wS, wO, 4, 5)
    close(ana, g["baked_weighted_grad"], rtol=1e-4, atol=1e-4 * scale)
    if "dense_weighted_grad" in g:
        ana = O.splat_grad_analytic(pts, sigma, ts, wS, wO, None, None)
        close(ana, g["dense_weighted_grad"], rtol=1e-4, atol=1e-4 * np.abs(g["dense_weighted_grad"]).max())
    # the in-tree pattern-optimisation loss: L1(baked_softor_2, baked_sum_2)  (transposed sum!)
    p = pts.clone().requires_grad_(True)
    S2 = O.baked_sum(p, sigma, ts, transposed=True)
    loss = O.l1_loss(O.baked_softor(p, sigma, ts), S2 if ts[0] == ts[1] else S2.T)
    loss.backward()
    close(loss.detach(), g["baked_l1"], rtol=1e-5)
    close(p.grad, g["baked_l1_grad"], rtol=1e-4, atol=1e-4 * np.abs(g["baked_l1_grad"]).max())


def test_kat1_survey_values(golden):
    """SURVEY.md Appendix B KAT1 literal values."""
    d = O.splat_dense(torch.tensor([[0.25, 0.75], [0.5, 0.5]]), 4.0, [8, 6])
    S, So = O.reduce_sum(d), O.softor(d)
    assert tuple(d.shape) == (2, 6, 8)
    close(S[3, 4], 1.0870383977890015, rtol=1e-6)
    close(S[4, 2], 1.2057127952575684, rtol=1e-6)
    close(So[4, 3], 0.9794197678565979, rtol=1e-6)
    assert So[3, 4].item() == 1.0
    close(S.sum(), 20.149953842163086, rtol=1e-6)
    close(So.sum(), 17.704214096069336, rtol=1e-6)


def test_windows_are_bit_exact_vs_reference_slices(golden):
    """Index outputs: the integer clip rectangles must reproduce the reference's slicing exactly --
    checked by re-building baked_sum from the windows with plain python slices."""
    g = golden("splat_small_rect")
    pts, sigma, ts = T(g["points"]), float(g["sigma"]), g["texture_size"].tolist()
    win = O.baked_windows(pts, sigma, ts, 4)
    fp, half = O.footprint_size(sigma, 4)
    assert (fp, half) == (13, 6)
    vals, _, _, _ = O._footprint_values(pts, sigma, ts, 4)
    tex = torch.zeros(ts[0], ts[1])
    for i in range(pts.shape[0]):
        (w0, s0, e0), (w1, s1, e1) = win[i, 0].tolist(), win[i, 1].tolist()
        tex[w0:w0 + e0 - s0, w1:w1 + e1 - s1] += vals[i, s0:e0, s1:e1]
    close(tex.T, g["baked_sum"], atol=1e-6)


def test_transforms(golden):
    g = golden("transforms")
    W = O.compose_world([1, 2, 3], [0.1, 0.2, 0.3], [2, 1, 0.5], [0.5, -0.5, 2.0], torch.eye(4), True)
    close(W, g["kat2_world"], rtol=1e-6, atol=1e-7)
    close(O.transform_points(T(g["kat2_verts"]), W), g["kat2_out"], rtol=1e-6, atol=1e-6)
    # SURVEY KAT2 literal
    close(W[0], [1.872586846, -0.159345075, 0.156495914, 1.5], rtol=1e-6)
    # seeded random draws, variates injected in the reference's draw order T, R, S
    mn, mx, u = T(g["rand_min"]), T(g["rand_max"]), T(g["rand_u"])
    for i in range(u.shape[0]):
        t, r, s = (O.uniform_between(mn[k], mx[k], u[i, k]) for k in range(3))
        W = O.compose_world(t, r, s, g["rand_centroid"], T(g["rand_world0"]), True)
        close(W, g["rand_worlds"][i], rtol=1e-5, atol=1e-6)
        close(O.transform_points(T(g["rand_verts"]), W), g["rand_outs"][i], rtol=1e-5, atol=1e-5)
    # parent/child chain, eval-mode rotation sequence from the EvalStepper
    st = O.EvalStepper([0, 0, -np.pi], [0, 0, np.pi], [0, 0, 0])
    for i in range(g["chain_rot"].shape[0]):
        r = st.sample()
        assert np.array_equal(r.numpy(), g["chain_rot"][i])
        a = O.compose_world([0, 0, 0], r, [1, 1, 1], [1, 0, 0], torch.eye(4), True)
        b = O.compose_world([0, 0, 0], [0, 0, 0], [1, 1, 1], [0, 2, 0], torch.eye(4), True)
        wa, wb = O.chain_world([a, b], [-1, 0])
        close(wa, g["chain_worlds"][i, 0], rtol=1e-6, atol=1e-7)
        close(wb, g["chain_worlds"][i, 1], rtol=1e-6, atol=1e-6)
        close(O.transform_points(T(g["chain_vb"]), wb), g["chain_child_verts"][i], rtol=1e-5, atol=1e-6)
    # non-mesh transformable with attribute draws
    u = T(g["tr_u"])
    for i in range(u.shape[0]):
        t = O.uniform_between(torch.tensor([0.0, -1.0, 0.0]), torch.tensor([0.0, 1.0, 0.0]), u[i, 0:3])
        r = O.uniform_between(torch.tensor([-0.3, 0.0, 0.0]), torch.tensor([0.3, 0.0, 0.0]), u[i, 3:6])
        W = O.compose_world(t, r, None, [0, 0, 0], T(g["tr_world0"]), False)
        close(W, g["tr_worlds"][i], rtol=1e-5, atol=1e-6)
        close(O.uniform_between(torch.tensor([1.0]), torch.tensor([3.0]), u[i, 6:7]), g["tr_power"][i], rtol=1e-6)
        close(O.uniform_between(torch.tensor([0.0, 0.1, 0.2]), torch.tensor([1.0, 0.9, 0.8]), u[i, 7:10]), g["tr_color"][i], rtol=1e-6)
        s = O.uniform_between(torch.tensor([0.1]), torch.tensor([10.0]), u[i, 10:11])
        close(s.repeat(3), g["tr_intensity"][i], rtol=1e-6)
    close(O.transform_points(T(g["tp_pts"]), T(g["tp_K"])), g["tp_out"], rtol=1e-5, atol=1e-6)
    close(O.transform_directions(T(g["tp_pts"]), T(g["rand_world0"])), g["td_out"], rtol=1e-5, atol=1e-6)
    close(O.build_projection_matrix(60, 0.01, 1000.0), g["tp_K"], rtol=1e-6)


def test_samplers_bit_exact(golden):
    g = golden("samplers")
    st = O.EvalStepper([0, 0, -np.pi], [0, 0, np.pi], [0, 0, 0])
    assert np.array_equal(np.stack([st.sample().numpy() for _ in range(12)]), g["eval_vec3"])
    st = O.EvalStepper([0.0], [0.05], [0.0])
    assert np.array_equal(np.stack([st.sample().numpy() for _ in range(14)]), g["eval_scalar"])
    st = O.EvalStepper([0.0, 1.0, -1.0], [0.035, 1.5, 0.0], [0.0, 1.0, -1.0])
    assert np.array_equal(np.stack([st.sample().numpy() for _ in range(12)]), g["eval_vec3_ranged"])
    st = O.EvalStepper([0.1], [10.0], [0.1])
    s2v = np.stack([st.sample().numpy().repeat(3) for _ in range(4)])
    assert np.array_equal(s2v, g["eval_s2v"])
    an = O.AnimationStepper(0, 5, 0, 5)
    assert [an.sample_eval() for _ in range(9)] == g["anim_eval"].tolist() == [0, 1, 2, 3, 4, 5, 0, 1, 2]
    rng = random.Random(1)
    assert [an.sample_train(rng) for _ in range(5)] == g["anim_train_seed1"].tolist()
    mn, mx = torch.tensor([-1.0, 0.0, 2.0]), torch.tensor([1.0, 0.5, 2.0])
    got = np.stack([O.uniform_between(mn, mx, T(u)).numpy() for u in g["train_uniform_u"]])
    assert np.array_equal(got, g["train_uniform"])


def test_laser(golden):
    g = golden("laser")
    rays = O.uniform_rays(0.0275, 18, 18)
    assert np.array_equal(rays.numpy(), g["rays"])
    K = T(g["K"])
    close(O.rays_to_ndc(rays, K), g["ndc"], rtol=1e-5, atol=1e-6)
    close(O.ndc_to_world(T(g["ndc"]), K), g["back"], rtol=1e-4, atol=1e-6)
    close(O.clamp_to_fov(T(g["wide"]), T(g["K01"])), g["wide_clamped"], rtol=1e-5, atol=1e-6)
    tex = O.splat_dense(O.rays_to_ndc(rays, K)[:, 0:2], 10.0, [64, 48]).sum(0)
    close(tex, g["gen_tex_sum"], rtol=1e-5, atol=1e-6)


def test_postprocess(golden):
    g = golden("postprocess")
    out = O.white_noise(g["img"], g["wn_noise"])
    assert np.array_equal(out, g["wn_out"])
    rng = random.Random(6)
    gates = [O.bernoulli_gates([0.5, 0.5], rng) for _ in range(16)]
    assert np.array_equal(np.array(gates), g["gates_seed6"])
    # blur: kornia is absent -> parity unpinned; check the restatement's own invariants
    k = O.gaussian_kernel1d(5, 3.0)
    close(k.sum(), 1.0, rtol=1e-6)
    assert torch.equal(k, k.flip(0))
    img = torch.rand(20, 31)
    const = torch.full((9, 11), 0.37)
    close(O.gaussian_blur2d(const, (3, 3), (5.0, 5.0)), const, rtol=1e-6)
    b = O.gaussian_blur2d(img, (5, 3), (2.0, 1.0))
    assert b.shape == img.shape
    # brute-force reflect reference
    ky, kx = O.gaussian_kernel1d(5, 2.0), O.gaussian_kernel1d(3, 1.0)
    H, W = img.shape

    def refl(i, n):
        return -i if i < 0 else (2 * (n - 1) - i if i >= n else i)

    for (r, c) in [(0, 0), (1, 30), (19, 15), (10, 0), (7, 9)]:
        acc = 0.0
        for a in range(5):
            for bb in range(3):
                acc += float(ky[a]) * float(kx[bb]) * float(img[refl(r + a - 2, H), refl(c + bb - 1, W)])
        close(b[r, c], acc, rtol=1e-5, atol=1e-6)


def test_oracle_equals_live_reference(golden):
    """Differential check on seeded inputs against the reference's outputs stored in ``tests/golden/live_reference.npz``
    (see its ``source``) and, when ``FIREFLIES_REF`` names a checkout of the original, against the reference executed here."""
    from oracle import make_golden
    sources = [("stored", golden("live_reference"))]
    if ref_loader.available():
        sources.append(("live", make_golden.live_reference_outputs(ref_loader.load())))
    for source, ref in sources:
        for i, (n, ts, sigma) in enumerate(make_golden.LIVE_CASES):
            c = f"c{i}_"
            pts = T(ref[c + "points"])
            assert pts.shape == (n, 2), source
            dense = O.splat_dense(pts, sigma, ts)
            st = int(ref.get(c + "dense_stride", 1))                     # the stored [40,64,96] stack keeps every other texel
            assert np.array_equal(dense.numpy()[:, ::st, ::st], ref[c + "dense"]), (source, i)
            close(O.baked_sum(pts, sigma, ts), ref[c + "baked_sum"], atol=1e-6)
            close(O.baked_sum(pts, sigma, ts, transposed=True), ref[c + "baked_sum_2"], atol=1e-6)
            close(O.baked_softor(pts, sigma, ts), ref[c + "baked_softor_2"], atol=1e-6)
            close(O.baked_sum(pts, sigma, ts, num_std=3), ref[c + "baked_sum_std3"], atol=1e-6)
            if ts[0] == ts[1]:   # the loop-over-points full-frame variants only work on square textures
                close(O.reduce_sum(dense), ref[c + "points_baked_sum"], atol=1e-5)
                close(O.softor(dense), ref[c + "points_baked_softor"], atol=1e-6)
        for j, a in enumerate(make_golden.LIVE_ANGLES):
            a32 = torch.tensor(a)        # the reference always receives an fp32 0-d tensor
            assert np.array_equal(O.yaw(a32).numpy(), ref["yaw"][j]), (source, a)
            assert np.array_equal(O.pitch(a32).numpy(), ref["pitch"][j]), (source, a)
            assert np.array_equal(O.roll(a32).numpy(), ref["roll"][j]), (source, a)


# ---- line / depth rasterisers (SURVEY 8(f) row 2) ---------------------------------------------------------
def test_lines_and_depth_match_reference_fixture(golden):
    g = golden("lines_depth")
    T = lambda a: torch.from_numpy(np.asarray(a))  # noqa: E731
    kat = O.rasterize_lines(T(g["kat3_lines"]), 4.0, [8, 6])
    assert kat.shape == (1, 6, 8)
    np.testing.assert_allclose(kat.numpy(), g["kat3"], rtol=1e-6, atol=1e-9)
    assert abs(float(kat[0, 1, 2]) - 0.9989765286) < 1e-6 and abs(float(kat.sum()) - 27.94803810) < 1e-4   # SURVEY App. B KAT3
    ts, sig = g["lines_ts"].tolist(), float(g["lines_sigma"])
    lines = T(g["lines"]).clone().requires_grad_(True)
    tex = O.rasterize_lines(lines, sig, ts)
    np.testing.assert_allclose(tex.detach().numpy(), g["lines_dense"], rtol=1e-6, atol=1e-9)
    S, So = tex.sum(dim=0), O.softor(tex)
    np.testing.assert_allclose(S.detach().numpy(), g["lines_sum"], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(So.detach().numpy(), g["lines_softor"], rtol=1e-6, atol=1e-9)
    ((S * T(g["lines_wS"])).sum() + (So * T(g["lines_wO"])).sum()).backward()
    ref = g["lines_weighted_grad"]
    np.testing.assert_allclose(lines.grad.numpy(), ref, rtol=1e-4, atol=1e-5 * np.abs(ref).max())
    pts = T(g["depth_points"])
    d = O.rasterize_depth(pts[:, 0:2], pts[:, 2:3], float(g["depth_sigma"]), g["depth_ts"].tolist())
    np.testing.assert_allclose(d.numpy(), g["depth_dense"], rtol=1e-6, atol=1e-9)
    for i, lv in enumerate(O.subsampled_point_raster(pts, 3, float(g["depth_sigma"]), g["depth_ts"].tolist())):
        np.testing.assert_allclose(lv.numpy(), g[f"depth_level{i}"], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(O.splat_dense_px(T(g["px_points"]), 6.0, [40, 24]).numpy(), g["px_dense"], rtol=1e-6, atol=1e-9)


def _perlin_angles(g, name):
    H, W, r0, r1, oc = g[f"{name}_cfg"].tolist()
    ang = torch.from_numpy(g[f"{name}_angles"])
    angles, f, off = [], 1, 0
    for _ in range(oc):
        n = (f * r0 + 1) * (f * r1 + 1)
        angles.append(ang[off:off + n].reshape(f * r0 + 1, f * r1 + 1)); off += n; f *= 2
    return [H, W], (r0, r1), oc, float(g[f"{name}_pers"]), angles


def test_perlin_matches_reference_fixture(golden):
    g = golden("perlin")
    for name in "abc":
        shape, res, oc, pers, angles = _perlin_angles(g, name)
        np.testing.assert_allclose(O.perlin_octaves(shape, res, oc, pers, angles).numpy(), g[f"{name}_noise"], rtol=1e-6, atol=1e-7)


# ---- NURBS-curve camera path, Poisson-disk initialisation, intersections ------------------------------------------
def test_nurbs_evaluator_known_answers():
    """geomdl is absent (parity unpinned): the restated evaluator is anchored on closed forms."""
    ctrl = [[0, 0, 0], [1, 2, 0], [3, 2, 1], [4, 0, 2]]
    kn = O.nurbs_normalize_knots([0, 0, 0, 0, 2, 2, 2, 2])                     # one Bezier segment -> Bernstein polynomials
    for t in (0.0, 0.3, 0.5, 0.99, 1.0):
        b = [(1 - t) ** 3, 3 * t * (1 - t) ** 2, 3 * t * t * (1 - t), t ** 3]
        want = [sum(b[i] * ctrl[i][d] for i in range(4)) for d in range(3)]
        close(O.nurbs_curve_point(ctrl, kn, 3, t), want, rtol=1e-14, atol=1e-15)
    s = np.sqrt(0.5)                                                           # rational quadratic quarter circle
    for t in np.linspace(0, 1, 17):
        p = O.nurbs_curve_point([[1, 0, 0], [1, 1, 0], [0, 1, 0]], [0, 0, 0, 1, 1, 1], 2, float(t), [1, s, 1])
        assert abs(p[0] ** 2 + p[1] ** 2 - 1.0) < 1e-14
    kn = O.nurbs_normalize_knots([0, 0, 0, 0, 1, 2, 2.5, 4, 4, 4, 4])            # partition of unity on a non-uniform vector
    assert kn[0] == 0.0 and kn[-1] == 1.0 and kn[5] == 0.5
    for t in np.linspace(0, 1, 41):
        span = O.nurbs_find_span(3, kn, 7, float(t))
        assert 3 <= span <= 6 and kn[span] <= t and (t < kn[span + 1] or t == 1.0)
        assert abs(sum(O.nurbs_basis(3, kn, span, float(t))) - 1.0) < 1e-14


@pytest.mark.parametrize("tag", ["bspline", "rational"])
def test_curve_pose_matches_reference_curve(golden, tag):
    """The reference's Curve.randomize / sample_rotation / sample_translation (run on the oracle evaluator) vs curve_pose."""
    g = golden("curve")
    kn = O.nurbs_normalize_knots(g["knots"])
    w = g["weights"] if tag == "rational" else None
    W = T(g[tag + "_W"])
    for d, want in zip(g[tag + "_deltas"], g[tag + "_worlds"]):
        assert np.array_equal(O.curve_pose(g["ctrl"], kn, 3, float(d), W, w).numpy(), want)
    pts = np.array([O.nurbs_curve_point(g["ctrl"], kn, 3, float(t), w) for t in np.linspace(0.0, 1.0, 101)])
    assert np.array_equal(pts, g[tag + "_points64"])
    d = g[tag + "_deltas"]
    assert np.all(d[:3] == 0.05) and abs(d[3] - 0.051) < 1e-12 and d[-3] == 0.05      # train quirk; eval walk; wrap at 1 - epsilon


def test_bridson_and_misc_match_reference(golden):
    g = golden("poisson_misc")
    np.random.seed(17)
    n, p = O.bridson(np.ones([48, 64]) * 5.5)
    assert n == int(g["uniform_n"]) and np.array_equal(p, g["uniform_pts"])
    np.random.seed(18)
    assert np.array_equal(O.bridson(g["varying_radius"], k=12)[1], g["varying_pts"])
    d = np.linalg.norm(p[:, None] - p[None], axis=-1) + np.eye(len(p)) * 1e9     # the property the sampler exists for
    assert d.min() > 5.5 * 0.7
    np.random.seed(19)
    _, s = O.bridson(np.ones([64, 48]) * O.poisson_radius(64, 48, 60))
    assert np.array_equal(O.blue_noise_rays(s, 64, 48, T(g["blue_K"])).numpy(), g["blue_rays"])
    t = O.ray_plane(T(g["rp_o"]), T(g["rp_d"]), T(g["rp_po"]), T(g["rp_pn"]))
    assert np.array_equal(t.numpy(), g["rp_t"], equal_nan=True)
    assert np.array_equal(O.sphere_sphere(T(g["ss_a"]), T(g["ss_ra"]), T(g["ss_b"]), T(g["ss_rb"])).numpy(), g["ss_hit"])
    close(O.rotation_matrix_from_vectors(T(g["rot_v1"]), T(g["rot_v2"])), g["rot"])
    close(O.rotation_matrix_from_vectors_with_fixed_up(T(g["rot_v1"]), T(g["rot_v2"])), g["rot_up"])


def test_product_poisson_sampler_consumes_the_numpy_stream_like_the_reference(golden):
    """Host-side set-up code of the product (numpy, like the reference): same draws, same points."""
    from fireflies_b200.sampling import poisson
    g = golden("poisson_misc")
    np.random.seed(17)
    n, p = poisson.bridson(np.ones([48, 64]) * 5.5)
    assert n == int(g["uniform_n"]) and np.array_equal(p, g["uniform_pts"])
    np.random.seed(18)
    assert np.array_equal(poisson.bridson(g["varying_radius"], k=12)[1], g["varying_pts"])
    np.random.seed(3)
    n, p = poisson.bridson(np.ones([20, 20]) * 4.0, k=8, radiusType="normDist")
    assert n == len(p) > 4


def test_nurbs_curve_object_host_logic(tmp_path):
    """Attribute checks and knot normalisation of the geomdl stand-in need no GPU; evaluating without one raises."""
    from fireflies_b200.utils.nurbs import NurbsCurve
    from fireflies_b200.utils.io import importBlenderNurbsObj
    c = NurbsCurve(device=torch.device("cpu"))
    with pytest.raises(ValueError):
        c.ctrlpts = [[0, 0, 0]] * 4                          # degree first
    c.degree = 3
    with pytest.raises(ValueError):
        c.ctrlpts = [[0, 0, 0]] * 3                          # needs degree + 1 points
    c.ctrlpts = [[0, 0, 0], [1, 2, 0], [3, 2, 1], [4, 0, 2], [5, 1, 1]]
    with pytest.raises(ValueError):
        c.knotvector = [0, 0, 0, 0, 1, 1, 1, 1]              # wrong length
    with pytest.raises(ValueError):
        c.knotvector = [0, 0, 0, 0, 3, 2, 4, 4, 4]           # decreasing
    c.knotvector = [0, 0, 0, 0, 2, 4, 4, 4, 4]
    assert c.knotvector == O.nurbs_normalize_knots([0, 0, 0, 0, 2, 4, 4, 4, 4]) and c.weights == [1.0] * 5
    with pytest.raises(ValueError):
        c.weights = [1, 1, 0, 1, 1]
    with pytest.raises(ValueError):
        NurbsCurve(9, [[0, 0, 0]] * 12, list(range(22)), device=torch.device("cpu"))
    obj = tmp_path / "path.obj"
    obj.write_text("# Blender\nv 0.0 0.0 0.0\nv 1.0 2.0 0.5\nv 3.0 2.5 -1.0\nv 4.0 0.0 2.0\ncstype bspline\ndeg 3\ncurv 0.0 1.0 1 2 3 4\n"
                   "parm u 0.0 0.0 0.0 0.0 1.0 1.0 1.0 1.0\nend\n")
    curve = importBlenderNurbsObj(str(obj), device=torch.device("cpu"))
    assert curve.degree == 3 and len(curve.ctrlpts) == 4 and curve.ctrlpts[2] == [3.0, 2.5, -1.0] and curve.knotvector[4] == 1.0
    with pytest.raises(ValueError):
        curve.evaluate_single(1.5)                           # outside the domain, like geomdl
    with pytest.raises(RuntimeError):
        curve.evaluate_single(0.5)                           # no CPU path


# ---- third-party arithmetic pinned against independent implementations that ARE in the image (VERDICT r01 item 4) -----------------
def test_silhouette_oracle_equals_reference_with_real_opencv(golden):
    """The reference's ApplySilhouette.post_process (apply_silhouette.py:17-40) executed with the real cv2.circle and its own
    random.randint draws (oracle/make_golden.py::post_cases; only kornia's blur is restated) against the oracle's analytic disc."""
    g = golden("postprocess")
    ones = np.ones((512, 448), dtype=np.float32)
    for i, (cx, cy, r) in enumerate(g["silhouette_discs"].tolist()):
        frame = g["silhouette_grad"] if i == 2 else ones
        close(O.silhouette(torch.from_numpy(frame), cx, cy, r), g["silhouette_out"][i], rtol=1e-6, atol=1e-7)
    # the filled cv2.circle itself is the analytic disc (x - cx)^2 + (y - cy)^2 <= r^2, also where it leaves the frame
    cv2 = pytest.importorskip("cv2")
    for cx, cy, r in [(150, 250, 200), (100, 300, 170), (380, 20, 60), (0, 0, 5), (447, 511, 33), (200, 200, 1), (37, 41, 0)]:
        m = cv2.circle(np.zeros((512, 448), np.float32), (cx, cy), r, color=1, thickness=-1)
        yy, xx = np.mgrid[0:512, 0:448]
        assert np.array_equal(m, (((xx - cx) ** 2 + (yy - cy) ** 2) <= r * r).astype(np.float32)), (cx, cy, r)


def test_blur_restatement_against_opencv_and_scipy():
    """oracle.gaussian_blur2d (kornia 0.7.1 restated: reflect border without edge repeat, separable, taps exp(-x^2 / 2 sigma^2) / sum)
    against cv2.GaussianBlur(BORDER_REFLECT_101) and scipy.ndimage.correlate1d(mode="mirror") for the three (kernel, sigma) pairs the
    reference uses (gauss_blur.py:18-28 callers: (3,3)/(5,5), main.py:69 (5,5)/(3,3), apply_silhouette.py:31 (11,11)/(5,5))."""
    cv2 = pytest.importorskip("cv2")
    ndi = pytest.importorskip("scipy.ndimage")
    img = np.random.default_rng(12).random((61, 47), dtype=np.float32)
    for (ky, kx), (sy, sx) in (((3, 3), (5.0, 5.0)), ((5, 5), (3.0, 3.0)), ((11, 11), (5.0, 5.0)), ((5, 3), (2.0, 1.0))):
        ours = O.gaussian_blur2d(torch.from_numpy(img), (ky, kx), (sy, sx)).numpy()
        for k, sg in ((ky, sy), (kx, sx)):          # taps: cv2.getGaussianKernel is the same normalised Gaussian
            close(O.gaussian_kernel1d(k, sg), cv2.getGaussianKernel(k, sg, cv2.CV_32F)[:, 0], rtol=1e-6, atol=1e-8)
        ocv = cv2.GaussianBlur(img, (kx, ky), sigmaX=sx, sigmaY=sy, borderType=cv2.BORDER_REFLECT_101)
        close(ours, ocv, rtol=1e-5, atol=1e-6)
        wy, wx = O.gaussian_kernel1d(ky, sy).double().numpy(), O.gaussian_kernel1d(kx, sx).double().numpy()
        sp = ndi.correlate1d(ndi.correlate1d(img.astype(np.float64), wx, axis=1, mode="mirror"), wy, axis=0, mode="mirror")
        close(ours, sp, rtol=1e-5, atol=1e-6)


def test_nurbs_evaluator_against_scipy_bspline():
    """oracle.nurbs_curve_point (geomdl 5.3.1 restated, entity/curve.py:52-53,74 call sites) against scipy.interpolate.BSpline on
    homogeneous control points: non-uniform knots, non-unit weights, degrees 2-4, parameters across every span."""
    BSpline = pytest.importorskip("scipy.interpolate").BSpline
    rng = np.random.default_rng(5)
    for degree, n in ((2, 5), (3, 7), (3, 12), (4, 9)):
        ctrl = rng.normal(size=(n, 3))
        w = rng.uniform(0.5, 2.0, size=n)
        inner = np.sort(rng.uniform(0.0, 1.0, size=n - degree - 1))
        knots = np.concatenate([np.zeros(degree + 1), inner, np.ones(degree + 1)])
        kn = O.nurbs_normalize_knots(knots.tolist())
        hom = np.concatenate([ctrl * w[:, None], w[:, None]], axis=1)
        spl = BSpline(np.asarray(kn), hom, degree)
        for t in np.concatenate([np.linspace(0.0, 1.0, 41)[:-1], inner, [0.999999]]):
            h = spl(float(t))
            close(O.nurbs_curve_point(ctrl.tolist(), kn, degree, float(t), w.tolist()), h[:3] / h[3], rtol=1e-12, atol=1e-13)
