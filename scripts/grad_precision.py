"""Dev helper: error of the backward kernels against an fp64 evaluation of the same gradient on the GPU (BASELINE config-3 shape, one sample;
baked_sum num_std 4 + baked_softor num_std 5, random upstream gradients).  Metric per component: |d - ref| / (1e-4 |ref| + 1e-4 ||ref_point||),
i.e. 1.0 = the tolerance the parity tests use."""
import os, sys
import torch
sys.path.insert(0, ".")
from fireflies_b200.graphics import rasterization as R

def ref64(pts, sigma, ts, gS, gO, H_s=20, H_o=25, R0=40):
    """fp64: per point a (2 R0 + 1)^2 crop; sum window |c - floor(P - H) - H| <= H per axis like the reference's slice."""
    dev = pts.device
    N = pts.shape[0]
    P = (pts.float() * torch.tensor([ts[0], ts[1]], device=dev, dtype=torch.float32)).double()      # fp32 product like the reference, then exact
    f = torch.floor((pts.float() * torch.tensor([ts[0], ts[1]], device=dev, dtype=torch.float32)) - 0.0)   # floor(P)
    off = torch.arange(-R0, R0 + 1, device=dev)
    ci = (f[:, 0].long().view(N, 1, 1) + off.view(1, 1, -1)).expand(N, 2 * R0 + 1, 2 * R0 + 1)
    ri = (f[:, 1].long().view(N, 1, 1) + off.view(1, -1, 1)).expand(N, 2 * R0 + 1, 2 * R0 + 1)
    ok = (ci >= 0) & (ci < ts[0]) & (ri >= 0) & (ri < ts[1])
    dc = ci.double() - P[:, 0].view(N, 1, 1)
    dr = ri.double() - P[:, 1].view(N, 1, 1)
    u = (dc * dc + dr * dr) / sigma
    g = torch.exp(-u * u) * ok
    def win(H):
        Pf = pts.float() * torch.tensor([ts[0], ts[1]], device=dev, dtype=torch.float32)
        o0 = torch.floor(Pf[:, 0] - H).long().view(N, 1, 1) + H
        o1 = torch.floor(Pf[:, 1] - H).long().view(N, 1, 1) + H
        return ((ci - o0).abs() <= H) & ((ri - o1).abs() <= H) & ok
    ms, mo = win(H_s), win(H_o)
    lin = (ri.clamp(0, ts[1] - 1) * ts[0] + ci.clamp(0, ts[0] - 1)).reshape(-1)
    logp = torch.zeros(ts[0] * ts[1], dtype=torch.float64, device=dev)
    logp.index_add_(0, lin, (torch.log1p(-(g * mo).clamp(max=1 - 1e-300))).reshape(-1))
    Pt = torch.exp(logp)
    excl = Pt[lin].view_as(g) / (1 - g * mo)
    coef = ms * gS.double().reshape(-1)[lin].view_as(g) + mo * gO.double().reshape(-1)[lin].view_as(g) * excl
    qv = coef * 4.0 * g * u / sigma
    return torch.stack([(qv * dc).sum((1, 2)) * ts[0], (qv * dr).sum((1, 2)) * ts[1]], 1)

torch.manual_seed(0)
N, ts, sigma = 4096, [2048, 2048], 100.0
gen = torch.Generator().manual_seed(0)
pts = (torch.rand(N, 2, generator=gen) * 0.96 + 0.02).cuda()
gS = torch.randn(ts[1], ts[0], device="cuda")
gO = torch.randn(ts[1], ts[0], device="cuda")
ref = ref64(pts, sigma, ts, gS, gO)
plan = R._SplatPlan(pts.unsqueeze(0).contiguous(), 1, sigma, ts[0], ts[1], 4, 5)
p1 = pts.unsqueeze(0).contiguous()
S_, O_ = plan.forward(p1, True, True, False)
tol = 1e-4 * ref.abs() + 1e-4 * ref.norm(dim=1, keepdim=True)
def report(name, d):
    e = (d.double() - ref).abs() / tol
    print(f"{name:22s}: max {float(e.max()):.4f}  rms {float((e * e).mean().sqrt()):.4f}  (tolerance units);  rel-to-norm {float((d.double() - ref).norm() / ref.norm()):.3e}")
variants = [("st rebuild", dict()), ("plain-load saved", dict(FFB_SPLAT_NO_TMA="1")), ("plain-load rebuild", dict(FFB_SPLAT_NO_TMA="1", NOSAVED="1")),
            ("general kernels", dict(GENERAL="1"))]
for name, kw in variants:
    os.environ.pop("FFB_SPLAT_NO_TMA", None)
    for k, v in kw.items():
        if k.startswith("FFB"): os.environ[k] = v
    if "GENERAL" in kw:
        os.environ["FFB_SPLAT_GENERAL"] = "1"
        pl = R._SplatPlan(p1, 1, sigma, ts[0], ts[1], 4, 5)
        d = pl.backward(p1, gS.unsqueeze(0).contiguous(), gO.unsqueeze(0).contiguous(), False)[0]
        del os.environ["FFB_SPLAT_GENERAL"]
    else:
        d = plan.backward(p1, gS.unsqueeze(0).contiguous(), gO.unsqueeze(0).contiguous(), False, None if "NOSAVED" in kw else O_)[0]
    report(name, d)
os.environ.pop("FFB_SPLAT_NO_TMA", None)
# the oracle's own fp32 autograd for scale
sys.path.insert(0, ".")
from oracle import ff_oracle as O
po = pts.cpu().clone().requires_grad_(True)
((O.baked_sum(po, sigma, ts) * gS.cpu()).sum() + (O.baked_softor(po, sigma, ts) * gO.cpu()).sum()).backward()
report("oracle fp32 autograd", po.grad.cuda())
