"""CPU: argument checks of the transform backward with the matrix gradient (ffb_transform_points_bwd_full,
ffb_transform_bwd_workspace_bytes) -- all decided before any device work -- and the refusal of CPU tensors."""
import pytest
import torch


@pytest.fixture(scope="module")
def nat():
    from fireflies_b200 import _build, _native
    _build.build()
    return _native


A, B, D, W = 1 << 20, 1 << 21, 1 << 22, 1 << 23        # distinct, never dereferenced addresses


def test_workspace_grows_with_the_point_count(nat):
    ws = nat.lib().ffb_transform_bwd_workspace_bytes
    sizes = [0, 1, 1024, 1025, 4099, 10 ** 5, 10 ** 6, 10 ** 7, 10 ** 9]
    got = [ws(v) for v in sizes]
    assert got[0] == 0 and got[1] == 0 and got[2] == 0            # one CTA: no partials, no workspace
    assert all(a <= b for a, b in zip(got, got[1:]))
    assert got[3] > 0 and got[-1] > got[3]
    assert got[-1] == got[-2]                                    # the partial count is capped: a fixed-size fold
    assert all(b % 64 == 0 for b in got)                         # 16 floats per partial


def test_workspace_query_rejects_negative_counts(nat):
    L = nat.lib()
    assert L.ffb_transform_bwd_workspace_bytes(-1) == 0
    assert b"V < 0" in L.ffb_last_error_string()


def call(nat, pts=A, V=4099, T=B, g=A + 64, d_pts=None, d_T=D, ws=W, nb=None):
    L = nat.lib()
    if nb is None:
        nb = L.ffb_transform_bwd_workspace_bytes(max(V, 0))
    return L.ffb_transform_points_bwd_full(pts, V, T, 0, g, d_pts, d_T, ws, nb, None)


@pytest.mark.parametrize("case", [dict(pts=None), dict(T=None), dict(g=None), dict(d_T=None), dict(V=-1), dict(V=-5, nb=0)])
def test_null_pointers_and_negative_counts(nat, case):
    assert call(nat, **case) == -1                               # FFB_E_ARG
    assert b"bad argument" in nat.lib().ffb_last_error_string()


def test_workspace_checks(nat):
    L = nat.lib()
    need = L.ffb_transform_bwd_workspace_bytes(4099)
    assert need > 0
    assert call(nat, ws=None) == -1                              # FFB_E_ARG: a workspace is needed
    assert b"null workspace" in L.ffb_last_error_string()
    assert call(nat, nb=need - 1) == -2                          # FFB_E_WORKSPACE
    assert b"too small" in L.ffb_last_error_string()
    assert call(nat, V=10 ** 7, nb=need) == -2


def test_cpu_tensors_have_no_path_when_the_transform_requires_grad():
    import fireflies_b200 as ff
    K = torch.eye(4, requires_grad=True)
    for f in (ff.utils.math.transform_points, ff.utils.math.transform_directions):
        with pytest.raises(RuntimeError, match="no CPU path"):
            f(torch.rand(5, 3), K)
        with pytest.raises(RuntimeError, match="no CPU path"):
            f(torch.rand(5, 3, requires_grad=True), K)
