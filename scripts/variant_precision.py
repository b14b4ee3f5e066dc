"""Dev helper: tolerance units (|d - ref| / (1e-4 |ref| + 1e-4 ||ref_point||)) of every backward variant against the fp64 closed form
on the data of tests/test_splat_gpu.py::test_every_kernel_variant."""
import os, sys
import torch
sys.path.insert(0, ".")
from oracle import ff_oracle as O
from fireflies_b200.graphics import rasterization as R
gen = torch.Generator().manual_seed(33)
B, N, ts, sigma = 2, 250, [288, 224], 36.0
pts = (torch.rand(B, N, 2, generator=gen) * 0.98 + 0.01)
wS = torch.randn(B, ts[1], ts[0], generator=gen)
wO = torch.randn(B, ts[1], ts[0], generator=gen)
for ns, no in ((4, 5), (0, 0), (3, 2)):
    for ws, wo in ((True, False), (False, True), (True, True)):
        anas = [O.splat_grad_analytic(pts[b], sigma, ts, wS[b] if ws else None, wO[b] if wo else None, ns or None, no or None) for b in range(B)]
        plan = R._SplatPlan(pts.cuda(), B, sigma, ts[0], ts[1], ns, no)
        s, o = plan.forward(pts.cuda(), ws, wo, False)
        for saved in ((None, o) if wo else (None,)):
            g = plan.backward(pts.cuda(), wS.cuda() if ws else None, wO.cuda() if wo else None, False, saved).cpu().double()
            worst = 0.0
            for b in range(B):
                ana = anas[b]; nrm = ana.norm(dim=1, keepdim=True)
                worst = max(worst, float(((g[b] - ana).abs() / (1e-4 * ana.abs() + 1e-4 * nrm + 1e-12)).max()))
            print(f"ns {ns} no {no} sum {int(ws)} softor {int(wo)} saved {saved is not None}: max {worst:.3f} tol units")
