"""The super-tile backward per candidate count of a 16x16 tile (st_tile: one candidate, two, three, four in one pass, five and
more with the product pass and the reciprocal), near and far candidates, against the fp64 reference; and PatternStep given one
[N,2] pattern for every sample, which bins it once.

Tile (1, 1) of super tile (1, 1) of a 256 x 64 texture at sigma 4 gets exactly k candidates.  The super-tile backward keeps a
candidate on a tile when the tile's nearest texel centre has g >= 1e-7 (distance^2 <= disc2) and calls it near when
distance^2 < near2 (wt_consts): near points sit inside the tile, far ones in a band 3.2 .. 3.8 texels left of it (inside tile 0
of the same super tile, where they are near)."""
import math

import numpy as np
import pytest
import torch

import test_splat_ref_gpu as T
from test_splat_ref_gpu import R  # noqa: F401  (fixture)

TS, SIGMA = [256, 64], 4.0
C0, R0 = 64, 16                           # super tile (1, 1)
DISC2, NEAR2 = SIGMA * math.sqrt(16.11809565095832), SIGMA * math.sqrt(5.545177444479562)


def tile_counts(P):
    """(candidates, near candidates) of each 16x16 tile of super tile (1, 1): st_stage's rule on points P (texels)."""
    cnt, near = [0] * 4, [0] * 4
    for px, py in P.tolist():
        px, py = px - C0, py - R0
        ry = max(-py, py - (T.WT - 1), 0.0)
        for i in range(4):
            rx = max(T.WT * i - px, px - (T.WT * i + T.WT - 1), 0.0)
            rr = rx * rx + ry * ry
            if rr <= DISC2:
                cnt[i] += 1
                near[i] += rr < NEAR2
    return cnt, near


def tile_pts(k, placement, seed):
    """k candidates of tile 1 (columns 80 .. 95, rows 16 .. 31), plus points in the rows below, clear of the super tile."""
    gen = torch.Generator().manual_seed(seed)
    nn = {"near": k, "far": 0, "mixed": (k + 1) // 2}[placement]
    u = torch.rand(k, 2, generator=gen, dtype=torch.float64)
    x = torch.where(torch.arange(k) < nn, 85.0 + 5.0 * u[:, 0], 76.2 + 0.6 * u[:, 0])
    y = 21.0 + 5.0 * u[:, 1]
    back = torch.rand(12, 2, generator=gen, dtype=torch.float64) * torch.tensor([TS[0] - 1.0, 20.0]) + torch.tensor([0.0, 40.0])
    P = torch.cat([torch.stack([x, y], 1), back])
    return T.texel_pts(P[torch.randperm(len(P), generator=gen)], TS), nn


FAMILY = {"stp": {"FFB_SPLAT_EAGER": "1"}, "st": {"FFB_SPLAT_EAGER": "0"}}


@pytest.mark.gpu
@pytest.mark.parametrize("sum_t", [False, True], ids=["natural", "transposed"])
@pytest.mark.parametrize("family", list(FAMILY))
@pytest.mark.parametrize("placement", ["near", "far", "mixed"])
@pytest.mark.parametrize("k", list(range(1, 9)))
def test_tile_candidate_counts(R, monkeypatch, k, placement, family, sum_t):
    pts = torch.stack([tile_pts(k, placement, seed=97 * k + 5 * b)[0] for b in range(T.B)])
    for b in range(T.B):
        cnt, near = tile_counts(T.scaled(pts[b], TS))
        assert cnt[1] == k and near[1] == tile_pts(k, placement, seed=97 * k + 5 * b)[1], (cnt, near)
    T.run_case(R, monkeypatch, pts, SIGMA, TS, 4, 5, sum_t=sum_t, env=FAMILY[family], seed=k)


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(FAMILY))
@pytest.mark.parametrize("k", [4, 5, 7])
def test_near_coincident_candidates(R, monkeypatch, k, family):
    """k points within 0.02 texels of one texel centre: g of each is within 1e-4 of 1, so every exclusive product is a
    product of small factors 1 - g."""
    gen = torch.Generator().manual_seed(k)
    P = torch.tensor([87.0, 23.0], dtype=torch.float64) + 0.02 * (torch.rand(k, 2, generator=gen, dtype=torch.float64) - 0.5)
    back = torch.rand(12, 2, generator=gen, dtype=torch.float64) * torch.tensor([TS[0] - 1.0, 20.0]) + torch.tensor([0.0, 40.0])
    pts = T.texel_pts(torch.cat([P, back]), TS)
    cnt, _ = tile_counts(T.scaled(pts, TS))
    assert cnt[1] == k
    T.run_case(R, monkeypatch, pts, SIGMA, TS, 4, 5, sum_t=True, batch=T.B, env=FAMILY[family], seed=k)


@pytest.mark.gpu
@pytest.mark.parametrize("fuse_loss", [False, True], ids=["upstream", "fused-l1"])
def test_pattern_step_bins_a_broadcast_pattern_once(monkeypatch, fuse_loss):
    """PatternStep given one [N,2] pattern: the same textures to the bit and the same pattern gradient as given the pattern
    copied per sample, from one binned instance instead of B."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import fireflies_b200 as ff
    R = ff.graphics.rasterization
    plans = []

    class Recording(R._SplatPlan):
        def __init__(self, points, *a, **k):
            super().__init__(points, *a, **k)
            plans.append((self.shared, self.ws.numel()))

    monkeypatch.setattr(R, "_SplatPlan", Recording)
    N, ts, B = 2048, (512, 512), 3
    gen = torch.Generator().manual_seed(3)
    pattern = (torch.rand(N, 2, generator=gen) * 0.96 + 0.02).cuda()
    gS = torch.randn(B, ts[0], ts[1], generator=gen).cuda()
    gO = torch.randn(B, ts[1], ts[0], generator=gen).cuda()
    step = ff.PatternStep(N, ts, 50.0, B, scene_batch=None, device="cuda", fuse_loss=fuse_loss)
    up = None if fuse_loss else (gS, gO)
    outs = []
    for p in (pattern.expand(B, N, 2).contiguous(), pattern):
        loss, dp, _ = step.forward_backward(p, upstream=up)
        outs.append((None if loss is None else loss.clone(), dp.clone(), step.last[0].clone(), step.last[1].clone()))
    torch.cuda.synchronize()
    (l_b, d_b, s_b, o_b), (l_s, d_s, s_s, o_s) = outs
    assert [sh for sh, _ in plans] == [False, True]
    assert plans[1][1] < plans[0][1]                      # one instance's lists instead of B
    assert torch.equal(s_s, s_b) and torch.equal(o_s, o_b)
    ref = d_b.cpu().numpy()
    np.testing.assert_allclose(d_s.cpu().numpy(), ref, rtol=1e-5, atol=1e-6 * float(np.abs(ref).max()))
    if fuse_loss:
        np.testing.assert_allclose(l_s.cpu().numpy(), l_b.cpu().numpy(), rtol=1e-6)
