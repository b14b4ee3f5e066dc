"""Time the batched Perlin textures against the per-scene loop they replace.

    python scripts/perlin_batch_time.py [--shape 1024] [--batches 32 256] [--iters 20] [--sequential-only]

Prints the card and its power limit, then per batch size: CUDA-event medians of ``perlin_texture_batch`` (drawn
parameters, three kernels) and of its first two kernels alone (octave sum into the noise buffer, no colour lerp), and a
host clock around B synchronised ``NoiseTextureLerpSampler.sample_train()`` calls (host draws included).  Rates are
given on the 12 B/texel of the output and on the 20 B/texel the kernels move (noise written and read back, output
written).  One JSON line per batch size.  ``--sequential-only`` times the per-scene loop alone (it runs on trees without
the batched entry point, so the loop can be compared across versions)."""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card() -> str:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                           stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ", power limit unknown"


def event_median(fn, iters: int, warmup: int = 3) -> float:
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times)


def sequential_ms(B: int, H: int, W: int, ca, cb) -> tuple:
    """Host clock around B synchronised sample_train() calls: median over a few repetitions, and the repetitions."""
    from fireflies_b200.sampling.noise_texture_lerp import NoiseTextureLerpSampler
    smp = NoiseTextureLerpSampler(ca, cb, [H, W])
    random.seed(3)
    torch.manual_seed(3)
    smp.sample_train()
    reps = max(1, min(5, 2000 // B))
    loop = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(B):
            smp.sample_train()
        torch.cuda.synchronize()
        loop.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(loop), reps


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", type=int, default=1024)
    ap.add_argument("--batches", type=int, nargs="+", default=[32, 256])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--sequential-only", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("perlin_batch_time.py needs a CUDA device")
    print("card:", card(), flush=True)
    H = W = args.shape
    ca, cb = torch.tensor([0.2, 0.5, 0.9], device="cuda"), torch.tensor([1.0, 0.0, 0.25], device="cuda")
    if args.sequential_only:
        for B in args.batches:
            ms_loop, reps = sequential_ms(B, H, W, ca, cb)
            print(json.dumps({"B": B, "shape": [H, W], "sequential_sample_train_ms": round(ms_loop, 2), "sequential_reps": reps}), flush=True)
        return
    from fireflies_b200 import _native as nat
    from fireflies_b200.sampling.noise_texture_lerp import perlin_texture_batch
    for B in args.batches:
        out = perlin_texture_batch((H, W), B, ca, cb, seed=1, sample0=0)
        step = [0]

        def batched():
            step[0] += B                                   # new samples every call: the drawn parameters vary
            perlin_texture_batch((H, W), B, ca, cb, seed=1, sample0=step[0], out=out)

        tex, d = out

        def noise_only():
            step[0] += B
            nat.check(nat.lib().ffb_perlin_texture_batch(B, H, W, 1, step[0], 0, None, None, 0, None, None, None, d.noise.data_ptr(),
                                                         d.minmax.data_ptr(), None, nat.stream()), "ffb_perlin_texture_batch")

        ms = event_median(batched, args.iters)
        ms_noise = event_median(noise_only, args.iters)
        ms_loop, reps = sequential_ms(B, H, W, ca, cb)
        texels = B * H * W
        rec = {"B": B, "shape": [H, W], "batched_ms": round(ms, 4), "textures_per_s": round(B / ms * 1e3, 1),
               "GBps_12B_per_texel": round(12 * texels / ms / 1e6, 1), "GBps_20B_per_texel": round(20 * texels / ms / 1e6, 1),
               "octave_sum_only_ms": round(ms_noise, 4), "lerp_share_ms": round(ms - ms_noise, 4),
               "sequential_sample_train_ms": round(ms_loop, 2), "sequential_reps": reps, "speedup": round(ms_loop / ms, 1),
               "store_vs_recompute": "recompute not built: not measured"}
        print(json.dumps(rec), flush=True)
        del out, tex, d


if __name__ == "__main__":
    main()
