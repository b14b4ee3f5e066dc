"""Dev helper: time the fused splat fwd / bwd at BASELINE config-3 shape (not the bench contract)."""
import os, sys, time
import torch
sys.path.insert(0, ".")
from fireflies_b200.graphics import rasterization as R

B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
N, ts = 4096, [2048, 2048]
gen = torch.Generator().manual_seed(0)
pts = (torch.rand(N, 2, generator=gen) * 0.96 + 0.02).cuda()
ptsB = pts.unsqueeze(0).repeat(B, 1, 1).contiguous()
plan = R._SplatPlan(ptsB, B, 100.0, ts[0], ts[1], 4, 5)
gS = torch.randn(B, ts[0], ts[1], device="cuda")
gO = torch.randn(B, ts[1], ts[0], device="cuda")
def t(fn, n=3):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n
hw = ts[0] * ts[1]
tp = t(lambda: R._SplatPlan(ptsB, B, 100.0, ts[0], ts[1], 4, 5))
tf = t(lambda: plan.forward(ptsB, True, True, True))
S_, O_ = plan.forward(ptsB, True, True, True)
res = {}
for name, eager in (("st_chunk8", "1"), ("st_oneshot", "0")):
    os.environ["FFB_SPLAT_EAGER"] = eager
    tb = t(lambda: plan.backward(ptsB, gS, gO, True, O_))
    res[name] = (tb, plan.backward(ptsB, gS, gO, True, O_))
    print(f"bwd {name:12s}: {tb:.3f} ms  ({B*8*hw/tb/1e6:.0f} GB/s algorithmic, frac {B*8*hw/tb/1e6/6458.4:.3f})")
os.environ.pop("FFB_SPLAT_EAGER", None)
ref = res["st_chunk8"][1]
d = res["st_oneshot"][1]
print(f"  st_oneshot vs st_chunk8: max|diff| {float((d - ref).abs().max()):.3e} of {float(ref.abs().max()):.3e}; rel-to-norm {float((d - ref).norm() / ref.norm()):.3e}")
# natural-layout sum gradient and single-reduction variants
gSn = gS.transpose(1, 2).contiguous()
for name, fn in [("nat sum+softor", lambda: plan.backward(ptsB, gSn, gO, False)), ("sum only T", lambda: plan.backward(ptsB, gS, None, True)),
                 ("softor only", lambda: plan.backward(ptsB, None, gO, False))]:
    print(f"bwd {name:15s}: {t(fn):.3f} ms")
tl = t(lambda: plan.backward_l1(ptsB, S_, O_, True))
print(f"fused L1 backward (st): {tl:.3f} ms ({B*8*hw/tl/1e6:.0f} GB/s algorithmic)")
tb = res["st_chunk8"][0]
print(f"B={B} prepare {tp:.3f} ms  fwd {tf:.3f} ms ({B*8*hw/tf/1e6:.0f} GB/s)  bwd {tb:.3f} ms ({B*8*hw/tb/1e6:.0f} GB/s)"
      f"  fwd+bwd per sample {(tf+tb)/B*1e3:.2f} us -> {B/(tf+tb)*1e3:.0f} samples/s, roofline frac {(B*(16*hw+16*N)/((tp+tf+tb)*1e-3))/6458.4e9:.3f}")
