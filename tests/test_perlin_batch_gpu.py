"""Batched Perlin material textures (``perlin_texture_batch`` / ``ffb_perlin_texture_batch``) and their use by ``SceneBatch``.

Injected samples must equal the single-texture path (``perlin_texture``, pinned to reference fixtures in
test_perlin_gpu.py) bit for bit; drawn samples must follow the Philox keying stated in include/ffb200.h, restated here in
numpy."""
import ctypes as C

import numpy as np
import pytest
import torch

import fake_mitsuba as fm

CA, CB = [0.2, 0.5, 0.9], [1.0, 0.0, 0.25]

# ---- include/ffb200.h, ffb_perlin_texture_batch, restated -----------------------------------------------------------------
_MASK = np.uint64(0xFFFFFFFF)
_M0, _M1, _W0, _W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
TAG_PARAMS, TAG_ANGLES = 0x9E700000, 0x9E710000


def philox(seed, c0, c1, c2, c3):
    """Philox4x32-10 on arrays of counters; returns the four output words as uint64 arrays holding 32-bit values."""
    c = [np.asarray(x, dtype=np.uint64) & _MASK for x in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    for _ in range(10):
        p0, p1 = _M0 * c[0], _M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK]
        k0, k1 = (k0 + _W0) & _MASK, (k1 + _W1) & _MASK
    return c


def drawn_params(seed, g, row):
    r = [int(x) for x in philox(seed, 0, g & 0xFFFFFFFF, g >> 32, TAG_PARAMS | row)]
    k = 1 + ((r[0] * 6) >> 32)
    octaves = 1 + ((r[1] * 4) >> 32)
    u53 = ((r[2] >> 5) * 67108864 + (r[3] >> 6)) / 9007199254740992.0
    return 2 ** k, octaves, 0.1 + 1.9 * u53


def drawn_angles(seed, g, row, res, octaves):
    """The per-octave lattices of sample g, in the layout perlin_angles returns."""
    sizes = [(res * 2 ** o + 1) for o in range(octaves)]
    n = np.arange(sum(s * s for s in sizes), dtype=np.uint64)
    w0 = philox(seed, n, g & 0xFFFFFFFF, g >> 32, TAG_ANGLES | row)[0]
    u = (w0 >> np.uint64(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)
    out, off = [], 0
    for s in sizes:
        out.append(torch.from_numpy(u[off:off + s * s].reshape(s, s).copy()))
        off += s * s
    return out


# ---- CPU: argument checks run before any device work ----------------------------------------------------------------------
def test_batch_argument_errors_do_not_need_a_gpu():
    from fireflies_b200 import _build, _native as nat
    _build.build()
    L = nat.lib()
    fake = C.c_void_p(16)          # never dereferenced: every call below is refused on the host
    args = lambda H, W, row=0, prm=None, ang=None, n=0: (4, H, W, 1, 0, row, prm, ang, n, fake, fake, fake, fake, fake, fake, None)  # noqa: E731
    assert L.ffb_perlin_texture_batch(*args(256, 512)) == -1
    assert b"multiples of 512" in L.ffb_last_error_string()
    assert L.ffb_perlin_texture_batch(*args(512, 512, row=1 << 16)) == -3
    assert L.ffb_perlin_texture_batch(*args(512, 512, ang=fake)) == -1
    prm = (nat.PerlinParams * 4)(*[nat.PerlinParams(8, 8, 2, 0, 0.5, 0)] * 4)
    n = 9 * 9 + 17 * 17
    assert L.ffb_perlin_texture_batch(*args(64, 64, prm=C.cast(prm, C.c_void_p), ang=fake, n=n - 1)) == -1   # angles too short
    assert b"past the end" in L.ffb_last_error_string()
    prm[2] = nat.PerlinParams(8, 8, 4, 0, 0.5, 0)                                                      # 8 * 2^3 does not divide 32
    assert L.ffb_perlin_texture_batch(*args(32, 32, prm=C.cast(prm, C.c_void_p), ang=fake, n=10 ** 6)) == -1
    prm[2] = nat.PerlinParams(8, 8, 9, 0, 0.5, 0)
    assert L.ffb_perlin_texture_batch(*args(4096, 4096, prm=C.cast(prm, C.c_void_p), ang=fake, n=10 ** 9)) == -1


# ---- GPU ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def S():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import fireflies_b200.sampling.noise_texture_lerp as S
    return S


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(512, 512), (512, 1024)])
def test_injected_samples_equal_the_single_texture_bit_for_bit(S, shape):
    params = [(2, 1, 0.5), (64, 4, 1.7), (8, 2, 0.3), (32, 3, 1.2), (4, 4, 0.9), (64, 1, 1.99), ((16, 2), 2, 0.75)]
    torch.manual_seed(5)
    angles = [S.perlin_angles(p[0] if isinstance(p[0], tuple) else (p[0], p[0]), p[1]) for p in params]
    tex, d = S.perlin_texture_batch(shape, len(params), CA, CB, seed=0, sample0=0, params=params, angles=angles)
    assert tex.shape == (len(params), 3) + shape
    ca, cb = torch.tensor(CA).cuda(), torch.tensor(CB).cuda()
    for b, (res, oc, pers) in enumerate(params):
        res = res if isinstance(res, tuple) else (res, res)
        noise1, tex1 = S.perlin_texture(shape, res, oc, pers, angles[b], ca, cb)
        assert torch.equal(d.noise[b], noise1), b
        assert torch.equal(tex[b], tex1), b
        assert tuple(d.res[b].tolist()) == res and int(d.octaves[b]) == oc and float(d.persistence[b]) == pers


@pytest.mark.gpu
def test_drawn_samples_follow_the_documented_keying(S):
    seed, sample0, row = 0x1234_5678_9ABC, (1 << 32) - 2, 3            # the sample index crosses a 32-bit word
    tex, d = S.perlin_texture_batch((512, 512), 4, CA, CB, seed=seed, sample0=sample0, row=row)
    ca, cb = torch.tensor(CA).cuda(), torch.tensor(CB).cuda()
    for b in range(4):
        g = sample0 + b
        res, oc, pers = drawn_params(seed, g, row)
        assert d.res[b].tolist() == [res, res] and int(d.octaves[b]) == oc and float(d.persistence[b]) == pers
        assert int(d.angle_offset[b]) == 0
        noise1, tex1 = S.perlin_texture((512, 512), (res, res), oc, pers, drawn_angles(seed, g, row, res, oc), ca, cb)
        assert torch.equal(d.noise[b], noise1), b
        assert torch.equal(tex[b], tex1), b


@pytest.mark.gpu
def test_drawn_samples_do_not_depend_on_the_split(S):
    whole, dw = S.perlin_texture_batch((512, 512), 16, CA, CB, seed=9, sample0=100, row=1)
    whole, raw = whole.clone(), dw.raw.clone()
    for q in range(4):
        part, dp = S.perlin_texture_batch((512, 512), 4, CA, CB, seed=9, sample0=100 + 4 * q, row=1)
        assert torch.equal(part, whole[4 * q:4 * q + 4]) and torch.equal(dp.raw, raw[4 * q:4 * q + 4])
    other_seed, _ = S.perlin_texture_batch((512, 512), 16, CA, CB, seed=10, sample0=100, row=1)
    other_row, _ = S.perlin_texture_batch((512, 512), 16, CA, CB, seed=9, sample0=100, row=2)
    for t in (other_seed, other_row):
        assert not any(torch.equal(t[b], whole[b]) for b in range(16))


@pytest.mark.gpu
def test_drawn_parameter_distributions_and_colour_range(S):
    B = 256
    tex, d = S.perlin_texture_batch((512, 512), B, CA, CB, seed=2024, sample0=0)
    k = torch.log2(d.res[:, 0].double()).round().long().cpu()
    assert torch.equal(d.res[:, 0], d.res[:, 1])
    # each of 6 (4) values: binomial(256, 1/6 (1/4)), within 5 standard deviations of the mean
    for vals, n in ((k, 6), (d.octaves.long().cpu(), 4)):
        cnt = torch.bincount(vals - 1, minlength=n)
        assert cnt.numel() == n and int(vals.min()) >= 1
        mu, sd = B / n, (B / n * (1 - 1 / n)) ** 0.5
        assert ((cnt.double() - mu).abs() <= 5 * sd).all(), cnt
    p = d.persistence.cpu()
    assert float(p.min()) >= 0.1 and float(p.max()) < 2.0
    assert abs(float(p.mean()) - 1.05) <= 5 * 1.9 / 12 ** 0.5 / B ** 0.5
    flat, nz = tex.reshape(B, 3, -1), d.noise.reshape(B, -1)
    lo, hi = nz.argmin(1), nz.argmax(1)
    for c in range(3):
        assert (flat[torch.arange(B), c, lo] == CA[c]).all() and (flat[torch.arange(B), c, hi] == CB[c]).all()
        assert (flat[:, c].amin(1) == min(CA[c], CB[c])).all() and (flat[:, c].amax(1) == max(CA[c], CB[c])).all()


def _texture_scene(ff, shape=(512, 512)):
    params = fm.FakeParams()
    params["mat-X.brdf_0.base_color.data"] = fm.TensorXf(torch.zeros(3, *shape))
    params["mat-X.brdf_0.roughness.value"] = fm.Float(0.5)
    sc = ff.Scene(params)
    mat = ff.material.Material("mat-X")
    mat.add_float_key("brdf_0.roughness.value", 0.1, 0.9)
    mat.add_vec3_sampler("brdf_0.base_color.data", ff.sampling.NoiseTextureLerpSampler(torch.tensor(CA), torch.tensor(CB), list(shape)))
    sc._materials.append(mat)
    return sc, params


@pytest.mark.gpu
def test_scene_batch_draws_texture_samplers(S):
    import fireflies_b200 as ff
    sc, params = _texture_scene(ff)
    sc.train()
    sb = sc.batch(seed=77)
    res = sb.randomize(4)
    tex = res.attribute("mat-X", "brdf_0.base_color.data")
    assert tex.shape == (4, 3, 512, 512) and tex.is_cuda
    assert res.attribute("mat-X", "brdf_0.roughness.value").shape == (4, 1)
    want, _ = S.perlin_texture_batch((512, 512), 4, CA, CB, seed=77, sample0=0, row=0)
    assert torch.equal(tex, want)
    res.write_sample(1)
    written = params["mat-X.brdf_0.base_color.data"]
    assert isinstance(written, fm.TensorXf) and written.t.is_cuda and torch.equal(written.t, tex[1])
    assert 0.1 <= float(params["mat-X.brdf_0.roughness.value"]) <= 0.9
    world, sampled = res.to_host()
    assert sampled.shape == (4, 1, 3)                                   # textures stay on the device
    ptr, before = tex.data_ptr(), tex.clone()
    noise_ptr = res.textures[("mat-X", "brdf_0.base_color.data")][1].noise.data_ptr()
    res2 = sb.randomize(4, out=res)
    tex2 = res2.attribute("mat-X", "brdf_0.base_color.data")
    assert res2 is res and tex2.data_ptr() == ptr and res.textures[("mat-X", "brdf_0.base_color.data")][1].noise.data_ptr() == noise_ptr
    assert not torch.equal(tex2, before)
    want, _ = S.perlin_texture_batch((512, 512), 4, CA, CB, seed=77, sample0=4, row=0)
    assert torch.equal(tex2, want)
    # eval mode and injected scalar variates: the texture rows still draw from Philox
    sc.eval()
    assert torch.equal(sc.batch(seed=77).randomize(4, sample0=4).attribute("mat-X", "brdf_0.base_color.data"), want)
    sc.train()
    inj = sc.batch(seed=77).randomize(4, sample0=4, variates=torch.full((4, 1, 3), 0.5, device="cuda"))
    assert torch.equal(inj.attribute("mat-X", "brdf_0.base_color.data"), want)
    assert torch.allclose(inj.attribute("mat-X", "brdf_0.roughness.value"), torch.full((4, 1), 0.5, device="cuda"))


@pytest.mark.gpu
def test_scene_batch_refuses_untileable_textures_and_samplers_without_a_record(S):
    import fireflies_b200 as ff
    sc, _ = _texture_scene(ff, (256, 256))
    with pytest.raises(ValueError, match="multiples of 512"):
        sc.batch()

    class Custom(ff.sampling.Sampler):
        _KIND = None
    sc, _ = _texture_scene(ff)
    sc._materials[0].add_float_sampler("brdf_0.custom", Custom(0.0, 1.0))
    with pytest.raises(NotImplementedError, match="no device record"):
        sc.batch()
