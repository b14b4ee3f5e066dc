"""The splat (fireflies_b200/csrc/ffb_splat.cu, ffb_splat_wt.cuh, ffb_splat_st.cuh) against a footprint-local fp64 reference,
for every kernel the dispatcher picks, at the list, chunk and texture-side edges where its kernels go wrong.

Every GPU case states which kernels it must launch: the names recorded by torch.profiler (CUDA activities) must equal what
`select` -- a Python mirror of the selection rules in ffb_splat.cu -- predicts, so a change in the selection fails by name instead
of silently leaving a kernel untested.  The case ids name the kernels and the reason they are chosen.

Tolerances (tests/test_splat_gpu.py): forward 1e-5 relative + 1e-6 absolute; gradients per component, 1e-4 relative + 1e-4 of
the point's own gradient norm (at least a tenth of the mean norm).  Every gradient check also requires a nonzero kernel gradient
for each point whose reference gradient norm is above 1e-12 of the largest, so a dropped gradient fails whatever its size."""
import math
import re

import numpy as np
import pytest
import torch

from oracle import ff_oracle as O

F64 = torch.float64
WT = 16                       # warp tile; super tiles are 4 WT x WT texels
WCH = 16                      # candidates a warp stages at once (longer super-tile lists go to the overflow kernels)
GTILE = (64, 32)              # CTA tile of the general kernels: columns, rows
B = 2


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import fireflies_b200.graphics.rasterization as R
    return R


# ---- mirror of the selection rules (make_plan, fill_raster, ffb_splat_fwd / _bwd / _bwd_l1) ----------------------------
class Sel:
    pass


def select(ts, sigma, N, ns, no, env=None):
    """What ffb_splat.cu decides for a call with these inputs; ``env``: the FFB_SPLAT_* variables set for it."""
    env = env or {}
    ts0, ts1 = ts
    sig = np.float32(sigma)
    root = math.floor(float(np.sqrt(sig)))               # floorf(sqrtf(sigma))

    def fp_of(k):
        f = root * k
        f += f % 2 == 0
        return f, (f - 1) // 2

    s = Sel()
    s.fp_s, s.half_s = fp_of(ns)
    s.fp_o, s.half_o = fp_of(no)
    s.h_s = max(1, math.ceil(math.sqrt(float(sig) * math.sqrt(87.0) * 1.02)))
    s.h_o = max(1, math.ceil(math.sqrt(float(sig) * math.sqrt(17.5) * 1.02)))
    s.H_s = s.half_s if ns > 0 else s.h_s
    s.mask_o = no > 0 and s.half_o < s.h_o
    s.H_o = s.half_o if s.mask_o else s.h_o
    s.h_union = max(s.H_s, s.H_o)
    fast_ok = (ns == 0 or (ts0 > s.fp_s and ts1 > s.fp_s)) and (no == 0 or (ts0 > s.fp_o and ts1 > s.fp_o))
    s.fast = fast_ok and ts0 <= 32000 and ts1 <= 32000 and env.get("FFB_SPLAT_GENERAL") != "1"
    s.no_tma = env.get("FFB_SPLAT_NO_TMA") == "1"
    s.msk = (s.H_s * s.H_s / float(sig)) ** 2 < 15.25
    wwin = 2.0 * max(s.H_s, s.H_o) + 1.0
    s.per_tile = N * (wwin + 4 * WT - 1) * (wwin + WT - 1) / (ts0 * ts1)
    s.eager = env["FFB_SPLAT_EAGER"] == "1" if "FFB_SPLAT_EAGER" in env else s.per_tile >= 2.0
    s.tw, s.th = ((4 * WT, WT) if s.fast else GTILE)
    s.tgx, s.tgy = -(-ts0 // s.tw), -(-ts1 // s.th)
    s.ts = ts
    return s


def tma_ok(sel, natural, transposed=False):
    """A tensor map needs its innermost side to be a multiple of 4 (16-byte rows): ts0 for natural [ts1, ts0] arrays, ts1 for
    the transposed sum."""
    ts0, ts1 = sel.ts
    return not sel.no_tma and (not natural or ts0 % 4 == 0) and (not transposed or ts1 % 4 == 0)


def fwd_expect(sel, S, O_, T):
    T, M = T and S, sel.mask_o and O_
    if not sel.fast:
        return {("splat_fwd_kernel", (S, O_, T))}
    fam = "splat_fwd_tma" if tma_ok(sel, O_ or (S and not T), S and T) else "splat_fwd_wt"
    return {(fam, (S, O_, T, M)), ("splat_fwd_ovf", (S, O_, T, M))}


def bwd_expect(sel, S, O_, T, V):
    T = T and S
    if not sel.fast:
        return {("splat_bwd_kernel", (S, O_, T))}
    tma = tma_ok(sel, O_ or (S and not T), S and T)
    if O_ and sel.mask_o and tma:
        return {("splat_bwd_tma", (S, True, T, V)), ("splat_bwd_ovf", (S, True, T, True, V, False))}
    if tma:
        K = S and sel.msk
        if sel.eager:
            return {("splat_bwd_stp", (S, O_, T, K, 0)), ("splat_bwd_ovf", (S, O_, T, False, False, False))}
        return {("splat_bwd_st", (S, O_, T, K)), ("splat_bwd_ovf", (S, O_, T, False, False, False))}
    M, V = O_ and sel.mask_o, V and O_
    return {("splat_bwd_wt", (S, O_, T, M, V)), ("splat_bwd_ovf", (S, O_, T, M, V, False))}


def loss_expect(sel, T):
    assert sel.fast and not sel.mask_o and tma_ok(sel, True, T)
    return {("splat_bwd_stp", (True, True, T, sel.msk, 1)), ("splat_bwd_ovf", (True, True, T, False, True, True))}


def expected(sel, reduce, sum_t, loss=False, saved=(False, True)):
    S, O_ = "sum" in reduce, "softor" in reduce
    want = fwd_expect(sel, S, O_, sum_t)
    if loss:
        return want | loss_expect(sel, sum_t)
    for v in (saved if O_ else (False,)):
        want |= bwd_expect(sel, S, O_, sum_t, v)
    return want


def kname(k):
    return f"{k[0]}<{','.join(str(int(a)) for a in k[1])}>"


def knames(ks):
    return "+".join(kname(k) for k in sorted(ks))


# ---- kernels launched, as recorded by torch.profiler ---------------------------------------------------------------------
_KERNEL = re.compile(r"\b(splat_[a-z_]+)<([^<>]*)>")


def parse_kernel(name):
    """'void ffb::splat::splat_bwd_stp<true, true, false, false, 0>(...)' or the integer form 'splat_bwd_stp<1, 1, 0, 0, 0>' ->
    ('splat_bwd_stp', (1, 1, 0, 0, 0)); None for kernels that are not splat kernels."""
    m = _KERNEL.search(name)
    if not m:
        return None
    args = []
    for a in m.group(2).split(","):
        a = {"true": "1", "false": "0"}.get(a.strip(), a.strip())
        v = re.search(r"(-?\d+)[uUlL]*$", a)
        assert v, f"cannot read template argument {a!r} of {name!r}"
        args.append(int(v.group(1)))
    return m.group(1), tuple(args)


def launched(fn):
    """Runs ``fn`` under torch.profiler with CUDA activities: (its result, names of the CUDA kernels it launched)."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]
    names += [k.name for e in prof.events() for k in getattr(e, "kernels", [])]
    assert names, "torch.profiler recorded no CUDA kernels: the launched kernels cannot be checked"
    return out, names


def splat_kernels(names):
    return set(filter(None, map(parse_kernel, names)))


def as_ints(ks):
    return {(k, tuple(int(a) for a in args)) for k, args in ks}


def test_parse_kernel_names():
    assert parse_kernel("splat_bwd_stp<1, 1, 1, 0, 0>") == ("splat_bwd_stp", (1, 1, 1, 0, 0))
    assert parse_kernel("void ffb::splat::splat_fwd_tma<true, false, true, false>(ffb::splat::RasterParams, "
                        "ffb::splat::WtConsts, CUtensorMap_st, CUtensorMap_st)") == ("splat_fwd_tma", (1, 0, 1, 0))
    assert parse_kernel("void ffb::splat::splat_bwd_stp<true, true, false, true, (ffb::splat::StMode)1>(...)") == \
        ("splat_bwd_stp", (1, 1, 0, 1, 1))
    assert parse_kernel("void ffb::splat::prepare_onepass_kernel<false>(ffb::splat::PrepParams)") is None
    assert parse_kernel("Memset (Device)") is None


# ---- footprint-local fp64 reference ----------------------------------------------------------------------------------------
def scaled(pts, ts):
    """P = float32(x) * ts in float32, as the kernels and the oracle form it."""
    return pts.detach().cpu().float() * torch.tensor([ts[0], ts[1]], dtype=torch.float32)


def ref_windows(pts, sigma, ts, num_std, h):
    """Half-open integer windows [lo, hi) per point and axis ([N, 2] each; empty = lo == hi == 0): the reference's baked clip
    rectangle (O.baked_windows) for num_std > 0, the square floor(P) +- h clipped to the texture for the dense semantics."""
    P = scaled(pts, ts)
    tsv = torch.tensor([ts[0], ts[1]])
    if num_std > 0:
        win = O.baked_windows(pts.detach().cpu(), sigma, ts, num_std).long()
        lo = win[:, :, 0]
        hi = torch.minimum(lo + (win[:, :, 2] - win[:, :, 1]).clamp(min=0), tsv)
    else:
        fl = torch.floor(P).long()
        lo, hi = (fl - h).clamp(min=0), torch.minimum(fl + h + 1, tsv)
    empty = (hi <= lo).any(dim=1, keepdim=True) | (lo >= tsv).any(dim=1, keepdim=True)
    return torch.where(empty, 0, lo), torch.where(empty, 0, hi)


def ref_splat(pts, sigma, ts, ns, no, wS=None, wO=None):
    """fp64 sum S and soft-OR O ([ts1, ts0]) of one pattern ``pts`` [N, 2] and, for upstream gradients wS / wO ([ts1, ts0] or
    None), d(<wS, S> + <wO, O>)/d pts [N, 2].  Evaluated over each point's window only: cost N x window area.  The dense
    semantics (num_std 0) use the square floor(P) +- h_s for both reductions (beyond it g < 1.7e-38)."""
    ts0, ts1 = ts
    sel = select(ts, sigma, pts.shape[0], ns, no)
    sig = float(np.float32(sigma))
    P = scaled(pts, ts).double()
    wins = [ref_windows(pts, sigma, ts, ns, sel.h_s), ref_windows(pts, sigma, ts, no, sel.h_s)]
    big = 1 << 30
    ulo = torch.minimum(*[torch.where(hi > lo, lo, big) for lo, hi in wins])
    uhi = torch.maximum(*[torch.where(hi > lo, hi, -big) for lo, hi in wins])
    live = (uhi > ulo).all(dim=1)
    ulo, uhi = torch.where(live[:, None], ulo, 0), torch.where(live[:, None], uhi, 0)
    W = (uhi - ulo).max(dim=0).values.clamp(min=1)
    cols = ulo[:, 0:1] + torch.arange(int(W[0]))                     # [N, W0]
    rows = ulo[:, 1:2] + torch.arange(int(W[1]))                     # [N, W1]

    def inside(lo, hi):
        return (((cols >= lo[:, 0:1]) & (cols < hi[:, 0:1]))[:, None, :] &
                ((rows >= lo[:, 1:2]) & (rows < hi[:, 1:2]))[:, :, None])

    ms, mo = inside(*wins[0]), inside(*wins[1])                      # [N, W1, W0]
    dc = (cols.double() - P[:, 0:1])[:, None, :]
    dr = (rows.double() - P[:, 1:2])[:, :, None]
    u = (dc * dc + dr * dr) / sig
    g = torch.exp(-(u * u))
    flat = rows.clamp(max=ts1 - 1)[:, :, None] * ts0 + cols.clamp(max=ts0 - 1)[:, None, :]
    S = torch.zeros(ts1 * ts0, dtype=F64).index_add_(0, flat[ms], g[ms])
    om = 1 - g
    nz, zero = mo & (om != 0), mo & (om == 0)
    prod = torch.ones(ts1 * ts0, dtype=F64).scatter_reduce_(0, flat[nz], om[nz], reduce="prod")
    zc = torch.zeros(ts1 * ts0, dtype=torch.long).index_add_(0, flat[zero], torch.ones(int(zero.sum()), dtype=torch.long))
    Ov = 1 - torch.where(zc > 0, 0.0, prod)
    grad = None
    if wS is not None or wO is not None:
        coef = torch.zeros_like(g)
        if wS is not None:
            coef = coef + ms * wS.double().flatten()[flat]
        if wO is not None:
            # prod_{m != n} (1 - g_m) from the product of the nonzero factors and the count of exact zeros (torch.prod's backward)
            pf, zf = prod[flat], zc[flat]
            excl = torch.where(zf == 0, pf / torch.where(om == 0, 1.0, om), torch.where((om == 0) & (zf == 1), pf, 0.0))
            coef = coef + mo * wO.double().flatten()[flat] * excl
        q = coef * 4.0 * g * u / sig
        grad = torch.stack([(q * dc).sum(dim=(1, 2)) * ts0, (q * dr).sum(dim=(1, 2)) * ts1], dim=1)
    return S.view(ts1, ts0), Ov.view(ts1, ts0), grad


@pytest.mark.parametrize("ns,no", [(4, 5), (0, 0), (3, 2)])
def test_reference_against_the_oracle(ns, no):
    """The footprint-local reference against the oracle's dense closed form (1e-12) and its float32 forwards."""
    gen = torch.Generator().manual_seed(40 + ns)
    ts, sigma = [96, 72], 16.0
    pts = torch.rand(40, 2, generator=gen) * 1.1 - 0.05
    pts[7] = pts[3]                                                     # a duplicate
    pts[9] = torch.tensor([30.0 / 96, 18.0 / 72])                       # on a texel centre: g = 1, an exact zero factor
    pts[10] = pts[9]                                                    # two of them
    wS, wO = torch.randn(ts[1], ts[0], generator=gen), torch.randn(ts[1], ts[0], generator=gen)
    S, Ov, G = ref_splat(pts, sigma, ts, ns, no, wS, wO)
    ana = O.splat_grad_analytic(pts, sigma, ts, wS, wO, ns or None, no or None)
    assert float((G - ana).abs().max()) <= 1e-12 * float(ana.abs().max())
    if ns:
        fwd_close(S, O.baked_sum(pts, sigma, ts, num_std=ns).double())
        fwd_close(Ov, O.baked_softor(pts, sigma, ts, num_std=no).double())
    else:
        d = O.splat_dense(pts, sigma, ts)
        fwd_close(S, O.reduce_sum(d).double())
        fwd_close(Ov, O.softor(d).double())
    for w, only in ((wS, "sum"), (wO, "softor")):       # one upstream gradient alone
        G1 = ref_splat(pts, sigma, ts, ns, no, w if only == "sum" else None, w if only == "softor" else None)[2]
        a1 = O.splat_grad_analytic(pts, sigma, ts, w if only == "sum" else None, w if only == "softor" else None, ns or None, no or None)
        assert float((G1 - a1).abs().max()) <= 1e-12 * float(a1.abs().max())


# ---- checks --------------------------------------------------------------------------------------------------------------
def ranges(idx):
    idx, out, i = [int(v) for v in idx], [], 0
    while i < len(idx):
        j = i
        while j + 1 < len(idx) and idx[j + 1] == idx[j] + 1:
            j += 1
        out.append(f"{idx[i]}..{idx[j]}" if j > i else f"{idx[i]}")
        i = j + 1
    return ", ".join(out)


def fwd_close(got, want, rtol=1e-5, atol=1e-6, what=""):
    got, want = got.detach().cpu().double(), want.detach().cpu().double()
    assert got.shape == want.shape, (got.shape, want.shape)
    err = (got - want).abs() - (atol + rtol * want.abs())
    worst = int(err.argmax())
    r, c = divmod(worst, got.shape[-1])
    assert not (err.max() > 0) and not err.isnan().any(), \
        f"{what}max violation {float(err.max()):.3e} at row {r} column {c}: got {float(got.flatten()[worst]):.9g}, " \
        f"want {float(want.flatten()[worst]):.9g}; {int((err > 0).sum())} texels off"


def grad_close(got, want, what=""):
    """close_grad of tests/test_splat_gpu.py plus the lost-gradient rule of tests/test_lines_ref_gpu.py."""
    got, want = got.detach().cpu().double(), want.detach().cpu().double()
    assert got.shape == want.shape and got.shape[-1] == 2, (got.shape, want.shape)
    nrm = want.norm(dim=1)
    lost = (nrm > 1e-12 * nrm.max()) & (nrm > 0) & (got == 0).all(dim=1)
    assert not lost.any(), f"{what}points with a nonzero reference gradient but an all-zero kernel gradient " \
                           f"({int(lost.sum())} of {got.shape[0]}): {ranges(lost.nonzero().flatten())}"
    scale = torch.maximum(nrm, 0.1 * nrm.mean())[:, None]
    err = (got - want).abs() - (1e-4 * want.abs() + 1e-4 * scale)
    worst = int(err.argmax())
    assert not (err.max() > 0) and not err.isnan().any(), \
        f"{what}max violation {float(err.max()):.3e} at point {worst // 2}: got {float(got.flatten()[worst]):.6e}, " \
        f"want {float(want.flatten()[worst]):.6e}, point norm {float(nrm[worst // 2]):.3e}"


# ---- one call of the splat, checked against the reference -----------------------------------------------------------
def set_env(monkeypatch, env):
    for k in ("FFB_SPLAT_GENERAL", "FFB_SPLAT_NO_TMA", "FFB_SPLAT_EAGER"):
        if k in env:
            monkeypatch.setenv(k, env[k])
        else:
            monkeypatch.delenv(k, raising=False)


def run_case(R, monkeypatch, pts, sigma, ts, ns, no, reduce=("sum", "softor"), sum_t=False, batch=None, env=None, loss=False,
             saved=(False, True), seed=0, loss_vs_unfused=False):
    """Forward, then the backward with and without the saved soft-OR output (or the fused L1 backward), of ``pts`` ([B, N, 2]
    per sample, or [N, 2] shared by ``batch`` samples), all against the fp64 reference, sample by sample; the splat kernels
    launched must be the ones `select` predicts.  ``loss_vs_unfused``: the fused L1 gradient against the plain backward given
    the same sign upstream gradients (tests/test_splat_gpu.py's rule) instead of fp64 -- for patterns of isolated points, whose
    L1 gradient is the float32 rounding of sum - soft-OR (a lone point's two terms cancel exactly)."""
    env = env or {}
    set_env(monkeypatch, env)
    shared = pts.dim() == 2
    Bn, N = (batch if shared else pts.shape[0]), pts.shape[-2]
    ws, wo = "sum" in reduce, "softor" in reduce
    sel = select(ts, sigma, N, ns, no, env)
    want = expected(sel, reduce, sum_t, loss, saved)
    gen = torch.Generator().manual_seed(seed)
    wS = torch.randn(Bn, ts[1], ts[0], generator=gen) if ws else None          # natural [ts1, ts0] orientation
    wO = torch.randn(Bn, ts[1], ts[0], generator=gen) if wo else None
    gs = (wS.transpose(1, 2) if sum_t else wS).contiguous().cuda() if ws else None
    go = wO.cuda() if wo else None
    p = pts.contiguous().cuda()
    plan = R._SplatPlan(p, Bn, sigma, ts[0], ts[1], ns, no)

    def call():
        s, o = plan.forward(p, ws, wo, sum_t)
        if loss:
            return s, o, [plan.backward_l1(p, s, o, sum_t)]
        return s, o, [plan.backward(p, gs, go, sum_t, o if v else None) for v in (saved if wo else (False,))]

    (s, o, grads), names = launched(call)
    got = splat_kernels(names)
    assert got == as_ints(want), f"launched {knames(got)}, expected {knames(want)} (all kernels: {sorted(set(names))})"
    for b in range(Bn):
        pb = pts if shared else pts[b]
        if loss:
            diff = o[b].cpu() - s[b].cpu()                 # mean |softor - sum (as stored)|, rasterization.py:589-599
            sg = torch.sign(diff) * np.float32(1.0 / (ts[0] * ts[1]))
            wsb, wob = -(sg.T if sum_t else sg), sg
        else:
            wsb, wob = (wS[b] if ws else None), (wO[b] if wo else None)
        S, Ov, G = ref_splat(pb, sigma, ts, ns, no, wsb, wob)
        if ws:
            fwd_close(s[b].T if sum_t else s[b], S, what=f"sample {b} sum: ")
        if wo:
            fwd_close(o[b], Ov, what=f"sample {b} soft-OR: ")
        if loss:
            lo, d = grads[0]
            fwd_close(lo[b:b + 1], diff.abs().double().mean().view(1), atol=1e-7, what=f"sample {b} loss: ")
            if loss_vs_unfused:
                gsb = (wsb.T if sum_t else wsb).contiguous()
                du = R._SplatPlan(pb.contiguous().cuda(), 1, sigma, ts[0], ts[1], ns, no).backward(
                    pb.contiguous().cuda(), gsb[None].cuda(), wob[None].contiguous().cuda(), sum_t)[0]
                assert not ((d[b] == 0).all(1) & (du != 0).any(1)).any(), f"sample {b}: fused L1 gradient lost"
                fwd_close(d[b], du, rtol=1e-4, atol=1e-5 * float(du.abs().max()), what=f"sample {b} loss gradient: ")
            else:
                grad_close(d[b], G, what=f"sample {b} loss gradient: ")
        else:
            for v, d in zip(saved if wo else (False,), grads):
                grad_close(d[b], G, what=f"sample {b} {'with' if v else 'without'} the saved soft-OR: ")
    return s, o, grads


def rand_pts(n, seed, lo=0.01, hi=0.99, shared=False):
    gen = torch.Generator().manual_seed(seed)
    return torch.rand(*(() if shared else (B,)), n, 2, generator=gen) * (hi - lo) + lo


def texel_pts(P, ts):
    """Points from texel positions: float32(P / ts), so that float32(x) * ts lands within an ulp of P."""
    return (torch.as_tensor(P, dtype=F64) / torch.tensor([ts[0], ts[1]], dtype=F64)).float()


# ---- 1. dispatch matrix --------------------------------------------------------------------------------------------------
REDUCE = {"both": ("sum", "softor"), "sum": ("sum",), "softor": ("softor",)}
COMBOS = [("both", False), ("both", True), ("sum", False), ("sum", True), ("softor", False)]


def dispatch_cases():
    """(id, kwargs of run_case) per case.  Per-sample points, B = 2, plus one shared-pattern run (batch = B) per family."""
    out = []

    def add(why, ts, sigma, N, ns, no, red, T, env=None, loss=False, shared=False):
        sel = select(ts, sigma, N, ns, no, env)
        want = expected(sel, REDUCE[red], T, loss)
        cid = (f"{why}-{ts[0]}x{ts[1]}-s{sigma:g}-n{N}-w{ns}{no}-{red}{'-T' if T else ''}{'-shared' if shared else ''}"
               f"{'-' + ','.join(f'{k[10:]}={v}' for k, v in sorted((env or {}).items())) if env else ''}->{knames(want)}")
        out.append(pytest.param(dict(ts=ts, sigma=sigma, N=N, ns=ns, no=no, red=red, T=T, env=env or {}, loss=loss,
                                     shared=shared), want, id=cid))

    dense, sparse = ([256, 192], 36.0, 120), ([512, 512], 36.0, 20)     # per_tile 9.2 / 0.29 (eager threshold 2)
    for why, (ts, sg, n) in (("tma-dense", dense), ("tma-sparse", sparse)):
        for red, T in COMBOS:
            add(why, ts, sg, n, 4, 5, red, T)                                # sum window exact at 4 std: K false
            if red != "softor":
                add(why + "-msk", ts, sg, n, 3, 5, red, T)                   # (H_s^2/sigma)^2 = 5.1 < 15.25: K true
        add(why, ts, sg, n, 4, 5, "both", False, shared=True)
    for red, T in COMBOS[:2] + COMBOS[4:]:
        add("tma-masko", *dense, 4, 2, red, T)                              # soft-OR window 13 < no-op radius 2*13+1: MASK_O
    add("tma-masko", *dense, 4, 2, "both", True, shared=True)
    for red, T in COMBOS:
        add("plain-sides2mod4", [258, 194], 36.0, 120, 4, 5, red, T)         # no side a multiple of 4: no tensor map
    for red, T in COMBOS[:2] + COMBOS[4:]:
        add("plain-sides2mod4-masko", [258, 194], 36.0, 120, 4, 2, red, T)
    add("plain-sides2mod4", [258, 194], 36.0, 120, 4, 2, "both", False, shared=True)
    add("plain-ts1-2mod4", [256, 194], 36.0, 120, 4, 5, "both", True)        # natural maps fine, transposed sum not
    add("plain-env", *dense, 4, 5, "both", False, env={"FFB_SPLAT_NO_TMA": "1"})
    for red, T in COMBOS:
        add("general-env", *dense, 4, 5, red, T, env={"FFB_SPLAT_GENERAL": "1"})
    add("general-env", *dense, 4, 5, "both", True, env={"FFB_SPLAT_GENERAL": "1"}, shared=True)
    add("general-small", [20, 16], 36.0, 12, 4, 5, "both", False)           # footprint 25 > 20: clipping is not an intersection
    add("general-small", [20, 16], 36.0, 12, 4, 5, "softor", False)
    for sg, K in ((36.0, "K0"), (48.0, "K1"), (120.0, "K1")):               # sum-window mask: (144/48)^2 = 9, (400/120)^2 = 11
        for T in (False, True):
            if sg == 120.0 and T:
                continue
            add(f"loss-{K}", [256, 256], sg, 120, 4, 5, "both", T, loss=True)
    add("loss-K1", [256, 256], 48.0, 120, 4, 5, "both", True, loss=True, shared=True)
    return out


DISPATCH = dispatch_cases()


@pytest.mark.gpu
@pytest.mark.parametrize("case,want", [p.values for p in DISPATCH], ids=[p.id for p in DISPATCH])
def test_dispatch(R, monkeypatch, case, want):
    c = case
    pts = rand_pts(c["N"], seed=len(c["red"]) + c["N"] + int(c["sigma"]), shared=c["shared"])
    run_case(R, monkeypatch, pts, c["sigma"], c["ts"], c["ns"], c["no"], REDUCE[c["red"]], c["T"],
             batch=B if c["shared"] else None, env=c["env"], loss=c["loss"], seed=c["N"])


FAMILIES = {"splat_fwd_tma": 8, "splat_fwd_wt": 8, "splat_fwd_kernel": 5, "splat_bwd_stp": 13, "splat_bwd_st": 9,
            "splat_bwd_tma": 6, "splat_bwd_wt": 14, "splat_bwd_kernel": 5}


def test_dispatch_matrix_reaches_every_instantiation():
    """The dispatch cases, as the selection mirror sees them, reach every instantiation of every family (splat_bwd_stp: 9 with
    given upstream gradients + 4 of the fused L1 loss mode)."""
    seen = set()
    for p in DISPATCH:
        seen |= p.values[1]
    for fam, n in FAMILIES.items():
        got = sorted(kname(k) for k in seen if k[0] == fam)
        assert len(got) == n, f"{fam}: {len(got)} of {n}: {got}"


# ---- 2. texture sides near the limits ----------------------------------------------------------------------------------
SIDES = [[30720, 32], [32000, 32], [32, 32000], [32001, 32], [65535, 16]]


def side_points(ts, sigma, ns, seed):
    """Along the long side: windows that start before, at and after texel 30000, windows straddling the far edge (one point
    just past it), a sweep over the last 3000 texels and a few near the start; across the short side spread over all rows
    (the last, partial super tile of a 32-wide texture included)."""
    a = 0 if ts[0] > ts[1] else 1
    L, Sh = ts[a], ts[1 - a]
    sel = select(ts, sigma, 1, ns, ns)
    H = sel.H_s
    longp = [30000 + H + d + 0.37 for d in (-9, -2, -1, 0, 1, 2, 9)]
    longp += [L - 1 - H + 0.5, L - 3.6, L - 0.4, L + 2.3, 5.2, 101.7, L / 2 + 0.21]
    longp += list(np.arange(L - 3000, L, 97.3) + 0.11)
    gen = torch.Generator().manual_seed(seed)
    shortp = (torch.rand(len(longp), generator=gen, dtype=F64) * (Sh + 1.0) - 0.5).tolist()
    P = [[lp, sp] if a == 0 else [sp, lp] for lp, sp in zip(longp, shortp)]
    return texel_pts(P, ts)


@pytest.mark.gpu
@pytest.mark.parametrize("ts", SIDES, ids=lambda t: f"{t[0]}x{t[1]}")
@pytest.mark.parametrize("ns,no", [(4, 5), (0, 0), (4, 2)], ids=["baked", "dense", "softor2"])
@pytest.mark.parametrize("red", ["both", "sum", "softor"])
def test_texture_sides(R, monkeypatch, ts, ns, no, red):
    """Sides up to the warp-tile path's 32000 and past it (general kernels, up to the ABI's 65535).  The warp-tile kernels mask
    the sum and the tight soft-OR windows with |c - f0| <= H around the window origin kept in the list entries; that origin
    must stay exact for windows starting at texel 30000 and beyond."""
    sigma = 36.0                                                     # footprints 25 / 31 / 13 < 32: baked windows on the warp-tile path
    pts = torch.stack([side_points(ts, sigma, ns, seed=1), side_points(ts, sigma, ns, seed=2)])
    for T in ((False, True) if ts == [32, 32000] and red != "softor" else (False,)):
        run_case(R, monkeypatch, pts, sigma, ts, ns, no, REDUCE[red], T, seed=ts[0] + ns)


@pytest.mark.gpu
def test_far_and_nan_points_contribute_nothing(R, monkeypatch):
    """Points far off a 32000-wide texture and NaN ones: outputs identical to the bit to those without them, gradients 0."""
    set_env(monkeypatch, {})
    ts, sigma = [32000, 32], 36.0
    pts = side_points(ts, sigma, 0, seed=3)
    far = torch.tensor([[2.0, 0.5], [1e4, 0.5], [-1e4, 0.5], [0.5, 1e6], [float("nan"), 0.5], [0.98, float("nan")]])
    for ns, no in ((4, 5), (0, 0), (4, 2)):
        outs = []
        for p in (pts, torch.cat([pts, far])):
            pc = p.cuda()
            plan = R._SplatPlan(pc, 1, sigma, ts[0], ts[1], ns, no)
            s, o = plan.forward(pc, True, True, False)
            g = torch.ones_like(o)
            outs.append((s, o, plan.backward(pc, g, g, False, o)))
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
        assert torch.equal(outs[1][2][0, len(pts):], torch.zeros(len(far), 2, device="cuda"))


# ---- 3. warp-tile list lengths across WCH ----------------------------------------------------------------------------
def candidates(P, sel, tile):
    """Candidates of super tile / CTA tile ``tile`` = (tx, ty): points whose binning window -- the union of the square
    floor(P) +- h_union and the reduction windows, clipped to the texture -- meets it."""
    ts0, ts1 = sel.ts
    fl = torch.floor(P).long()
    lo = (fl - sel.h_union).clamp(min=0)
    hi = torch.minimum(fl + sel.h_union + 1, torch.tensor([ts0, ts1]))
    x0, y0 = tile[0] * sel.tw, tile[1] * sel.th
    hit = (lo[:, 0] < x0 + sel.tw) & (hi[:, 0] > x0) & (lo[:, 1] < y0 + sel.th) & (hi[:, 1] > y0) & (hi > lo).all(1)
    return int(hit.sum())


def crowd(k, ts, tile, tsz, margin, nback, seed):
    """``k`` points whose binning windows (half width ``margin``) lie inside tile ``tile`` of size ``tsz``, plus ``nback``
    points in the rows below it, clear of it."""
    gen = torch.Generator().manual_seed(seed)
    x0, y0 = tile[0] * tsz[0], tile[1] * tsz[1]
    inner = torch.rand(k, 2, generator=gen, dtype=F64) * torch.tensor([tsz[0] - 2 * margin - 1.0, tsz[1] - 2 * margin - 1.0],
                                                                          dtype=F64) + torch.tensor([x0 + margin, y0 + margin], dtype=F64)
    yb = y0 + tsz[1] + margin
    back = torch.rand(nback, 2, generator=gen, dtype=F64) * torch.tensor([ts[0] - 1.0, ts[1] - 1 - yb], dtype=F64) + \
        torch.tensor([0.0, yb], dtype=F64)
    P = torch.cat([inner, back])
    return texel_pts(P[torch.randperm(len(P), generator=gen)], ts)


WT_FAMILY = {"stp": ((4, 5), {"FFB_SPLAT_EAGER": "1"}, False), "st": ((4, 5), {"FFB_SPLAT_EAGER": "0"}, False),
             "tma": ((4, 2), {}, False), "wt": ((4, 5), {"FFB_SPLAT_NO_TMA": "1"}, False), "loss": ((4, 5), {}, True)}


@pytest.mark.gpu
@pytest.mark.parametrize("shared", [False, True], ids=["persample", "shared3"])
@pytest.mark.parametrize("family", list(WT_FAMILY))
@pytest.mark.parametrize("k", [15, 16, 17, 40])
def test_warp_tile_list_lengths(R, monkeypatch, k, family, shared):
    """Super tile (1, 1) of a 256 x 64 texture with exactly k candidates, across WCH = 16 (the binning hands lists longer than
    WCH to the overflow kernels; splat_bwd_st stages them in rounds).  At sigma 4 the binning window is floor(P) +- 5, so
    points with floor(P) in columns 5..58 and rows 5..10 of the super tile are candidates of it alone.  Shared patterns run
    with B = 3 (the overflow kernels decode the sample of an item as it / count)."""
    (ns, no), env, loss = WT_FAMILY[family]
    ts, sigma = [256, 64], 4.0
    sel = select(ts, sigma, k + 20, ns, no, env)
    assert sel.fast and sel.h_union <= 5
    nb = 3 if shared else B
    pts = torch.stack([crowd(k, ts, (1, 1), (64, 16), 5, 20, seed=100 * k + b) for b in range(nb)])
    for b in range(nb):
        assert candidates(scaled(pts[b], ts), sel, (1, 1)) == k
    if shared:
        pts = pts[0]
    run_case(R, monkeypatch, pts, sigma, ts, ns, no, sum_t=False, batch=nb if shared else None, env=env, loss=loss, seed=k,
             loss_vs_unfused=loss)


# ---- 4. general-path list lengths across CHUNK = 128 and KCACHE = 6 ------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shared", [False, True], ids=["persample", "shared"])
@pytest.mark.parametrize("red", ["both", "sum", "softor"])
@pytest.mark.parametrize("k", [127, 128, 129, 300])
def test_general_list_lengths(R, monkeypatch, k, red, shared):
    """CTA tile (1, 1) of the general kernels (64 x 32) with exactly k candidates: across the 128-record staging chunk, and the
    backward's record reload for the second pass when a tile has more than one chunk.  Every warp block (8 rows x 32
    columns) sees far more than the 6 candidates whose g the backward caches."""
    env = {"FFB_SPLAT_GENERAL": "1"}
    ts, sigma = [192, 96], 4.0
    sel = select(ts, sigma, k + 20, 4, 5, env)
    assert not sel.fast and sel.h_union <= 5
    pts = torch.stack([crowd(k, ts, (1, 1), GTILE, 5, 20, seed=7 * k + b) for b in range(B)])
    for b in range(B):
        assert candidates(scaled(pts[b], ts), sel, (1, 1)) == k
    run_case(R, monkeypatch, pts[0] if shared else pts, sigma, ts, 4, 5, REDUCE[red], sum_t=red != "softor",
             batch=B if shared else None, env=env, seed=k)


# ---- 5. item decode of the chunked super-tile backward, super-tile borders ------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("ts,nb", [([256, 64], 2), ([320, 48], 3)], ids=["grid4x4-pow2", "grid5x3-B3-ragged"])
def test_chunked_backward_item_decode(R, monkeypatch, ts, nb):
    """splat_bwd_stp walks chunks of 8 consecutive (super tile, sample) items: by shifts on a power-of-two super-tile grid, by
    division otherwise (here 15 super tiles x 3 samples = 45 items: a ragged last chunk of 5)."""
    sel = select(ts, 16.0, 60, 4, 5)
    tgx, tiles = sel.tgx, sel.tgx * sel.tgy
    pow2 = tgx & (tgx - 1) == 0 and tiles & (tiles - 1) == 0
    assert pow2 == (ts == [256, 64]) and (pow2 or (tiles * nb) % 8 != 0) and sel.eager
    gen = torch.Generator().manual_seed(nb)
    pts = torch.rand(nb, 60, 2, generator=gen) * 0.98 + 0.01
    for red, T in COMBOS:
        run_case(R, monkeypatch, pts, 16.0, ts, 4, 5, REDUCE[red], T, seed=T + nb)


@pytest.mark.gpu
@pytest.mark.parametrize("ts", [[200, 76], [202, 74]], ids=["200x76-tma", "202x74-plain"])
@pytest.mark.parametrize("ns,no", [(4, 5), (4, 2), (0, 0)], ids=["baked", "softor2", "dense"])
def test_super_tile_borders(R, monkeypatch, ts, ns, no):
    """Windows straddling super-tile borders (columns = 0 mod 64, rows = 0 mod 16) on textures whose sides are not multiples
    of 64 or 16, for the TMA-fed and the plain kernels."""
    P = [[64 * i + d, 16 * j + e] for i in range(4) for j in range(5) for d, e in ((0.3, -0.4), (-0.6, 0.2), (3.7, 2.1))]
    P += [[ts[0] - 0.3, 16 * j + 7.5] for j in range(5)] + [[64 * i + 31.2, ts[1] - 0.45] for i in range(4)]
    base = texel_pts(P, ts)
    pts = torch.stack([base, base.flip(0)])
    for red, T in COMBOS:
        run_case(R, monkeypatch, pts, 9.0, ts, ns, no, REDUCE[red], T, seed=ts[0])
