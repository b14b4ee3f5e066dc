"""CPU: argument checks of the blur adjoint (ffb_blur_bwd) and of the differentiable ``gaussian_blur2d`` -- all decided before
any device work, so they need no GPU."""
import ctypes as C

import pytest
import torch


@pytest.fixture(scope="module")
def nat():
    from fireflies_b200 import _build, _native
    _build.build()
    return _native


def desc(nat, B=1, H=32, W=32, k=(5, 5), s=(3.0, 3.0), noise=0):
    return nat.PostDesc(B, H, W, k[0], k[1], s[0], s[1], noise, 0.0, 0.0, 0, 0)


A, G = 1 << 20, 1 << 30          # two distinct, never dereferenced addresses


@pytest.mark.parametrize("case,code,msg", [
    (dict(g_out=None), -1, b"null"),
    (dict(g_in=None), -1, b"null"),
    (dict(d=None), -1, b"null"),
    (dict(k=(4, 5)), -1, b"odd"),
    (dict(k=(5, 6)), -1, b"odd"),
    (dict(H=2), -1, b"kernel/2"),
    (dict(W=5, k=(5, 11)), -1, b"kernel/2"),
    (dict(noise=1), -1, b"noise"),
    (dict(g_in=A), -1, b"alias"),
    (dict(g_in=A + 4 * 32 * 32 - 4), -1, b"alias"),       # overlapping ranges
    (dict(k=(17, 5)), -3, b"15"),
    (dict(k=(5, 17)), -3, b"15"),
    (dict(k=(0, 5)), -1, b"blur stage"),
    (dict(s=(0.0, 1.0)), -1, b"sigma"),
    (dict(B=0), -1, b"positive"),
])
def test_blur_bwd_argument_errors(nat, case, code, msg):
    lib = nat.lib()
    kw = {k: case[k] for k in ("B", "H", "W", "k", "s", "noise") if k in case}
    d = C.byref(desc(nat, **kw)) if case.get("d", 1) is not None else None
    rc = lib.ffb_blur_bwd(d, case.get("g_out", A), case.get("g_in", G), None)
    assert rc == code
    assert msg in lib.ffb_last_error_string()


def test_gaussian_blur2d_refuses_what_it_does_not_implement(nat):
    from fireflies_b200.postprocessing import gaussian_blur2d
    x = torch.rand(1, 1, 16, 16)
    with pytest.raises(RuntimeError, match="no CPU path"):
        gaussian_blur2d(x, (5, 5), (3.0, 3.0))
    with pytest.raises(ValueError, match="border_type"):
        gaussian_blur2d(x, (5, 5), (3.0, 3.0), border_type="constant")
    with pytest.raises(NotImplementedError):
        gaussian_blur2d(x, (5, 5), torch.tensor([[3.0, 3.0]]))
    with pytest.raises(NotImplementedError):
        gaussian_blur2d(x, 5, (torch.tensor(3.0), 3.0))


def test_blur_spec_reads_kornia_style_arguments():
    from fireflies_b200.postprocessing.gauss_blur import blur_spec
    assert blur_spec(5, 3) == ((5, 5), (3.0, 3.0))
    assert blur_spec((5, 3), [2.0, 1.5]) == ((5, 3), (2.0, 1.5))
    with pytest.raises(ValueError):
        blur_spec((5, 5, 5), 1.0)
