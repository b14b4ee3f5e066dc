"""Dev helper: the config-3 step through PatternStep vs hand-assembled, per-phase CUDA-event times."""
import os, sys, json
import torch
sys.path.insert(0, ".")
import fireflies_b200 as ff
from fireflies_b200.graphics import rasterization as R
import bench
B = 256
dev = torch.device("cuda", 0)
g0 = torch.Generator().manual_seed(0)
pattern = (torch.rand(4096, 2, generator=g0) * 0.96 + 0.02).to(dev)
ptsB = pattern.unsqueeze(0).repeat(B, 1, 1).contiguous()
gS = torch.randn(B, 2048, 2048, device=dev); gO = torch.randn(B, 2048, 2048, device=dev)
scene = bench.build_scene(ff, dev); sb = scene.batch(seed=1)
step = ff.PatternStep(4096, (2048, 2048), 100.0, B, scene_batch=sb, device=dev)
def run(tag, rnd, **env):
    os.environ.pop("FFB_SPLAT_EAGER", None)
    os.environ.update(env)
    ms = []
    for i in range(8):
        m = {}
        step.forward_backward(pattern, upstream=(gS, gO), sample0=i * B, marks=m, randomize=rnd)
        torch.cuda.synchronize()
        if i >= 3: ms.append([m[a].elapsed_time(m[b]) for a, b in (("start", "prepare"), ("prepare", "fwd"), ("fwd", "bwd"), ("bwd", "end"), ("start", "end"))])
    t = torch.tensor(ms).mean(0).tolist()
    print(f"{tag:34s} prepare {t[0]:.3f} fwd {t[1]:.3f} bwd {t[2]:.3f} fold {t[3]:.3f} total {t[4]:.3f}")
run("PatternStep + randomize", True)
run("PatternStep, no randomize", False)
run("PatternStep + randomize, one-shot", True, FFB_SPLAT_EAGER="0")
run("PatternStep, no randomize, one-shot", False, FFB_SPLAT_EAGER="0")
os.environ.pop("FFB_SPLAT_EAGER", None)
# hand-assembled like the round-1 bench
ev = lambda: torch.cuda.Event(enable_timing=True)
for rnd in (True, False):
    acc = []
    side = torch.cuda.Stream()
    for i in range(8):
        e = [ev() for _ in range(5)]
        cur = torch.cuda.current_stream()
        e[0].record()
        if rnd:
            side.wait_stream(cur)
            with torch.cuda.stream(side): sb.randomize(B, sample0=i * B)
        plan = R._SplatPlan(ptsB, B, 100.0, 2048, 2048, 4, 5); e[1].record()
        _, so = plan.forward(ptsB, True, True, True); e[2].record()
        d = plan.backward(ptsB, gS, gO, True, so); e[3].record()
        cur.wait_stream(side)
        dp = R.reduce_over_samples(d); e[4].record()
        torch.cuda.synchronize()
        if i >= 3: acc.append([e[j].elapsed_time(e[j + 1]) for j in range(4)] + [e[0].elapsed_time(e[4])])
    t = torch.tensor(acc).mean(0).tolist()
    print(f"{'hand-assembled, randomize=' + str(rnd):34s} prepare {t[0]:.3f} fwd {t[1]:.3f} bwd {t[2]:.3f} fold {t[3]:.3f} total {t[4]:.3f}")
print("--- no synchronize between steps")
for rnd in (True, False):
    allm = []
    for i in range(12):
        m = {}
        step.forward_backward(pattern, upstream=(gS, gO), sample0=i * B, marks=m, randomize=rnd)
        allm.append(m)
    torch.cuda.synchronize()
    print("randomize", rnd, "bwd per step:", " ".join(f"{m['fwd'].elapsed_time(m['bwd']):.2f}" for m in allm), "| fwd:", " ".join(f"{m['prepare'].elapsed_time(m['fwd']):.2f}" for m in allm[:6]),
          "| step:", " ".join(f"{m['start'].elapsed_time(m['end']):.2f}" for m in allm[:6]))
print("--- bench-like loops, 10 steps back to back, with the NVML clock sampler")
def hand(i):
    cur = torch.cuda.current_stream(); side = step._side
    side.wait_stream(cur)
    with torch.cuda.stream(side): sb.randomize(B, sample0=i * B)
    plan = R._SplatPlan(ptsB, B, 100.0, 2048, 2048, 4, 5)
    _, so = plan.forward(ptsB, True, True, True)
    d = plan.backward(ptsB, gS, gO, True, so)
    cur.wait_stream(side)
    return R.reduce_over_samples(d)
for rep in range(2):
    for tag, fn in (("PatternStep", lambda i: step.forward_backward(pattern, upstream=(gS, gO), sample0=i * B)), ("hand-assembled", hand)):
        for i in range(3): fn(i)
        torch.cuda.synchronize()
        cs = bench.ClockSampler(0); cs.start()
        e0, e1 = ev(), ev(); e0.record()
        for i in range(10): fn(3 + i)
        e1.record(); torch.cuda.synchronize()
        c = cs.stop()
        print(f"{tag:16s} {e0.elapsed_time(e1) / 10:.3f} ms/step  clocks {c}")
