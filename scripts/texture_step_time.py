"""Times the projector-texture backward on the GPU it runs on (CUDA events, warm-up, medians) and prints one JSON object.

1. ``ffb_blur_bwd`` against the forward blur (``ffb_postprocess`` with a blur stage only) on 64 x 1024^2 frames (256 MiB in
   and out: larger than L2) for k = 3, 5, 11, the two alternated window by window in the same run.  Both read 4 B and write
   4 B per texel, so their ratio compares like with like.
2. ``TextureStep.backward`` at configs[1]'s shape (18x18 rays, 500^2, sigma 10, (5,5)/(3,3) blur, B = 32) and at B = 256,
   2048^2 (same rays), with the algorithmic bytes and their rate as a fraction of the HBM bandwidth measured by a device
   copy in the same run.

The card's name and power limit are read in the same run (``nvidia-smi`` query).  Writes nothing unless ``--out`` is given.

    python scripts/texture_step_time.py [--windows 7] [--iters 20] [--out result.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + " (power limit not readable)"


def time_ms(fn, iters):
    """Mean time per call over ``iters`` back-to-back calls, CUDA events."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def hbm_peak_gbs(iters):
    x = torch.empty(2 << 30, dtype=torch.uint8, device="cuda")
    y = torch.empty_like(x)
    for _ in range(3):
        y.copy_(x)
    ms = min(time_ms(lambda: y.copy_(x), iters) for _ in range(3))
    return 2 * x.numel() / ms / 1e6


def blur_pair(nat, k, windows, iters):
    B, H, W = 64, 1024, 1024
    x = torch.rand((B, H, W), device="cuda")
    y = torch.empty_like(x)
    g = torch.rand((B, H, W), device="cuda")
    gi = torch.empty_like(g)
    d = nat.PostDesc(B, H, W, k, k, k / 2.0, k / 2.0, 0, 0.0, 0.0, 0, 0)
    L, st = nat.lib(), nat.stream()

    def fwd():
        nat.check(L.ffb_postprocess(C.byref(d), x.data_ptr(), None, None, y.data_ptr(), st), "ffb_postprocess")

    def bwd():
        nat.check(L.ffb_blur_bwd(C.byref(d), g.data_ptr(), gi.data_ptr(), st), "ffb_blur_bwd")
    for _ in range(5):
        fwd()
        bwd()
    f, b = [], []
    for _ in range(windows):
        f.append(time_ms(fwd, iters))
        b.append(time_ms(bwd, iters))
    fm, bm = statistics.median(f), statistics.median(b)
    gbs = 8 * B * H * W / 1e6
    return {"k": k, "frames": [B, H, W], "fwd_ms": round(fm, 4), "bwd_ms": round(bm, 4), "bwd_over_fwd": round(bm / fm, 3),
            "fwd_gbs": round(gbs / fm, 1), "bwd_gbs": round(gbs / bm, 1),
            "bwd_over_fwd_per_window": [round(bb / ff, 3) for ff, bb in zip(f, b)]}


def texture_step(ff, O, B, ts, windows, iters, peak):
    rays = O.uniform_rays(0.0275, 18, 18)
    A = torch.tensor([[0.5, 0.0, 0.0, 0.5], [0.0, 0.5, 0.0, 0.5], [0.0, 0.0, 1.0, 0.0], [0.0, 0.0, 0.0, 1.0]])
    K = (A @ O.build_projection_matrix(60, 0.01, 1000.0)).cuda()
    laser = ff.projection.Laser(ff.entity.Transformable("projector"), rays.cuda(), K, 60.0, 0.01, 1000.0)
    step = ff.TextureStep(laser, sigma=10.0, texture_size=ts, blur=((5, 5), (3.0, 3.0)))
    step.texture()
    g = torch.randn((B, ts[1], ts[0], 3), device="cuda")
    for _ in range(3):
        step.backward(g)
    runs = [time_ms(lambda: step.backward(g), iters) for _ in range(windows)]
    ms = statistics.median(runs)
    texels = ts[0] * ts[1]
    # the upstream gradients read once (12 B / texel / sample); one frame: channel extraction (12 B read + 4 B written),
    # blur adjoint (8 B), splat backward (4 B read); the fold's partial sums and the [N,3] vectors are not counted
    nbytes = 12 * B * texels + (16 + 8 + 4) * texels
    gbs = nbytes / ms / 1e6
    return {"rays": rays.shape[0], "texture": ts, "B": B, "sigma": 10.0, "ms": round(ms, 4), "algorithmic_bytes": nbytes,
            "gbs": round(gbs, 1), "fraction_of_measured_hbm_peak": round(gbs / peak, 3)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("texture_step_time.py needs a CUDA device")
    import fireflies_b200 as ff
    from fireflies_b200 import _native as nat
    from oracle import ff_oracle as O
    res = {"card": card()}
    peak = hbm_peak_gbs(a.iters)
    res["hbm_copy_gbs"] = round(peak, 1)
    res["blur"] = [blur_pair(nat, k, a.windows, a.iters) for k in (3, 5, 11)]
    res["texture_step"] = [texture_step(ff, O, 32, [500, 500], a.windows, a.iters, peak),
                           texture_step(ff, O, 256, [2048, 2048], a.windows, max(a.iters // 4, 3), peak)]
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
