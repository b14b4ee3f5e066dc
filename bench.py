#!/usr/bin/env python
"""bench.py -- pattern-optimisation scene samples/sec on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload = BASELINE.json configs[2] ("batched pattern optimisation": 4096 laser points into a 2048x2048
projector texture, 256 randomised scenes per step, fwd+bwd); with N GPUs every rank runs 256 scenes per step
(weak scaling; N=8 is configs[4], 2048 scenes/step) and the only collective is the allreduce of the [4096,2]
pattern gradient.  One step = fireflies_b200.PatternStep.forward_backward(pattern, upstream=...):
randomise B scenes (sampling + 4x4 compose + 100k-vertex transform), bin + splat forward (baked_sum_2 +
baked_softor_2 semantics), splat backward against resident upstream texture gradients, fold the per-sample
gradients, allreduce.  With N > 1 the run starts with parallel.multi_gpu_selfcheck (`multi_gpu_check` in the line;
a mismatch exits non-zero).  `side` carries the other single-GPU configs (configs[0] step latency, configs[1],
configs[3]).

Prints ONE JSON line (rank 0).  `value` is device-timed with all inputs resident in HBM; `e2e` is the same step
through the public API (fireflies_b200.PatternStep.step_host) with HOST buffers for the pattern, the loss and the
gradient.  `cpu_baseline` / `--impl reference` time the CPU port of the reference algorithm (oracle/) on the host.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

N_POINTS, TS, SIGMA, V_MESH = 4096, (2048, 2048), 100.0, 100_000
METRIC = "pattern-opt scene samples/sec (splat fwd+bwd + randomize)"
UNIT = "scene samples/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="scene samples per step per GPU")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side", action="store_true", help="skip the side measurements of the other single-GPU configs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy; with N GPUs "
                         "rank 0 writes the allreduced gradient of the whole step and its own shard of the scene samples")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def config(batch, world):
    return {"workload": "configs[2] batched pattern optimisation (configs[4] when n_gpus=8)", "points": N_POINTS,
            "texture": list(TS), "sigma": SIGMA, "reductions": "baked_sum_2(num_std=4,transposed)+baked_softor_2(num_std=5)",
            "scenes_per_step_per_gpu": batch, "scenes_per_step": batch * world, "mesh_vertices": V_MESH,
            "mesh_randomisation": "translate+rotate+scale ranged, train mode (Philox)",
            "parallelism": f"dp{world} over scene samples; allreduce of d(points) [4096,2]",
            "l2": "inputs larger than L2 (per step 4 x 4.3 GB of textures/gradients vs 126 MB L2); no flush needed"}


# ---------------------------------------------------------------------------------------------------
# clocks (nvidia-smi recipe of B200_PROFILING.md, sampled through NVML during the timed region)
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown",
               0x100: "display_clock_setting"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self._stop, self._t, self._go = [], set(), None, threading.Event(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    def _run(self):
        # Sampling starts when the main thread has enqueued the timed steps (go()): the device then still has all but the first
        # fraction of a step in front of it, so every sample is taken under load, and no NVML call (a driver round trip of up to
        # milliseconds) competes with the kernel launches of the first timed step, where the host is not yet ahead of the device
        # (this was not the cause of the stalled steps of DESIGN.md 6 -- the caching allocator was -- but it keeps the driver out of
        # the launch path of the step where a host delay reaches the device).
        self._go.wait()
        while True:                                          # at least one sample, however short the timed region
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            if self._stop.wait(0.005):
                break

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def go(self):
        self._go.set()

    def stop(self):
        if self._t is not None:
            self._go.set()
            self._stop.set()
            self._t.join()
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference algorithm (test infrastructure used only as the timed baseline)
# ---------------------------------------------------------------------------------------------------
def cpu_scene_step(O, pts, gS, gO, verts, gen):
    """One scene sample on the CPU: randomise (T,R,S draw + compose + vertex transform), baked_sum_2 + baked_softor_2
    forward, backward to the points against the upstream gradients."""
    u = torch.rand(3, 3, generator=gen)
    t = O.uniform_between(torch.tensor([-0.5, -0.5, -0.5]), torch.tensor([0.5, 0.5, 0.5]), u[0])
    r = O.uniform_between(torch.tensor([-3.1, -3.1, -3.1]), torch.tensor([3.1, 3.1, 3.1]), u[1])
    s = O.uniform_between(torch.tensor([0.5, 0.5, 0.5]), torch.tensor([2.0, 2.0, 2.0]), u[2])
    W = O.compose_world(t, r, s, [0.0, 0.0, 0.0], torch.eye(4), True)
    v = O.transform_points(verts, W)
    p = pts.clone().requires_grad_(True)
    S = O.baked_sum(p, SIGMA, list(TS), transposed=True)
    So = O.baked_softor(p, SIGMA, list(TS))
    ((S * gS).sum() + (So * gO).sum()).backward()
    return p.grad, v


def cpu_inputs():
    g = torch.Generator().manual_seed(0)
    pts = torch.rand(N_POINTS, 2, generator=g) * 0.96 + 0.02
    g4 = torch.Generator().manual_seed(4)
    gS, gO = torch.randn(TS[0], TS[1], generator=g4), torch.randn(TS[1], TS[0], generator=g4)
    verts = torch.rand(V_MESH, 3, generator=torch.Generator().manual_seed(1)) * 2 - 1
    return pts, gS, gO, verts


def run_cpu(n_scenes, warm=1):
    from oracle import ff_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    pts, gS, gO, verts = cpu_inputs()
    gen = torch.Generator().manual_seed(2)
    for _ in range(warm):
        cpu_scene_step(O, pts, gS, gO, verts, gen)
    t0 = time.perf_counter()
    for _ in range(n_scenes):
        cpu_scene_step(O, pts, gS, gO, verts, gen)
    dt = time.perf_counter() - t0
    return n_scenes / dt, cores, dt


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ff_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    pts, gS, gO, verts = cpu_inputs()
    gen = torch.Generator().manual_seed(2)
    per_step = 1                                  # bounded sample: one scene of the 256-scene step per "step"
    for _ in range(args.warmup):
        cpu_scene_step(O, pts, gS, gO, verts, gen)
    t0 = time.perf_counter()
    for _ in range(args.steps * per_step):
        cpu_scene_step(O, pts, gS, gO, verts, gen)
    dt = time.perf_counter() - t0
    val = args.steps * per_step / dt
    sample = f"{per_step} scene sample of the step's {args.batch} per step (full 4096-point / 2048^2 / 100k-vertex size)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config(args.batch, 1),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU port of the reference algorithm (oracle/ff_oracle.py, vectorised scatter form of baked_sum_2/"
                "baked_softor_2 + torch autograd) on all host threads; the reference itself is pure Python and cannot "
                "travel to the GPU box"}))


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
class _Params(dict):
    def update(self, *a, **k):
        if a or k:
            return super().update(*a, **k)


def build_scene(ff, device):
    verts = torch.rand(V_MESH, 3, generator=torch.Generator().manual_seed(1)) * 2 - 1
    sc = ff.Scene(_Params(), device=device)
    m = ff.entity.Mesh("mesh-Bench", verts.to(device), device)
    c = lambda v: torch.tensor(v, device=device)  # noqa: E731
    m.translate(c([-0.5, -0.5, -0.5]), c([0.5, 0.5, 0.5]))
    m.rotate(c([-3.1, -3.1, -3.1]), c([3.1, 3.1, 3.1]))
    m.scale(c([0.5, 0.5, 0.5]), c([2.0, 2.0, 2.0]))
    sc._meshes.append(m)
    sc.train()
    return sc


DUMP_SUBSET = 1 << 20       # elements kept of an array larger than this: 4 MB each, about 13 MB for the whole dump


def dump_outputs(dirname, dp, res, textures):
    """Write what one PatternStep.forward_backward call returned as float32 ``<dirname>/<name>.npy``: the pattern gradient
    ``dpoints`` [N,2] and the randomised ``world`` [B,E,4,4] and ``sampled`` [B,S,3] whole; of the transformed ``vertices``
    [B,V,3] and of the step's textures (``PatternStep.last``: ``sum_texture`` [B,ts0,ts1], ``softor_texture`` [B,ts1,ts0]) the
    elements at DUMP_SUBSET flat indices drawn, sorted, from torch.Generator().manual_seed(0) (``*_subset``, 1-D) when the
    array is larger than that.  Same arguments, same inputs: two builds can be compared file by file.  With N ranks this is
    rank 0's call: ``dpoints`` is allreduced over the step's B*N samples, everything else belongs to rank 0's B samples only,
    so only dumps taken with the same number of ranks compare."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    arrays = {"dpoints": dp, "world": res.world, "sampled": res.sampled, "vertices": res.vertices,
              "sum_texture": textures[0], "softor_texture": textures[1]}
    for name, t in arrays.items():
        if t.numel() > DUMP_SUBSET:
            idx = torch.randint(0, t.numel(), (DUMP_SUBSET,), generator=torch.Generator().manual_seed(0)).sort().values
            t, name = t.reshape(-1)[idx.to(t.device)], name + "_subset"
        np.save(os.path.join(dirname, name + ".npy"), t.detach().float().cpu().numpy())


def side_configs(ff, device, peak):
    """The other single-GPU BASELINE configs, as short side measurements (CUDA events, medians; inputs resident; a 256 MB buffer is
    rewritten between iterations so that nothing is served from L2).  Not the headline metric."""
    from fireflies_b200.graphics import rasterization as R
    from fireflies_b200.postprocessing.base import run_postprocess
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)

    def timed(fn, n=10, do_flush=True):
        for _ in range(3):
            fn()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for a, b in ev:
            if do_flush:
                flush.zero_()
            a.record(); fn(); b.record()
        torch.cuda.synchronize()
        t = sorted(a.elapsed_time(b) for a, b in ev)
        return t[len(t) // 2]

    out = {}
    # ---- configs[0]: the reference's own loop (rasterization.py:583-607): 100 points -> 512^2, L1(softor, sum), one sample, plus a
    #      single mesh with rotate_z randomised (examples/01_hello_world.py:23-33).  Launch-bound: eager API vs the captured graph.
    g0 = torch.Generator().manual_seed(0)
    p0 = (torch.rand(100, 2, generator=g0) * 0.8 + 0.1).to(device)
    sc0 = ff.Scene(_Params(), device=device)
    m0 = ff.entity.Mesh("mesh-One", (torch.rand(10_000, 3, generator=g0) * 2 - 1).to(device), device)
    m0.rotate_z(-3.14159, 3.14159)
    sc0._meshes.append(m0)
    sc0.train()
    sb0 = sc0.batch(seed=9)
    step0 = ff.PatternStep(100, (512, 512), 100.0, 1, scene_batch=None, device=device)
    replay = step0.capture(p0)
    side = torch.cuda.Stream(device=device)

    def graphed():
        cur = torch.cuda.current_stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            sb0.randomize(1)
        replay(p0)
        cur.wait_stream(side)

    def eager():
        q = p0.clone().requires_grad_(True)
        m0.randomize(); m0.get_randomized_vertices()
        s, o = R.splat_reduce(q, 100.0, [512, 512], sum_transposed=True)
        R.l1_loss(o, s).backward()

    n_wall = 200
    for fn_name, fn in (("graph", graphed), ("eager_reference_api", eager)):
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n_wall):
            fn()
        torch.cuda.synchronize()
        out.setdefault("config0_step_ms", {})[fn_name] = (time.perf_counter() - t0) / n_wall * 1e3
    out["config0_step_ms"]["splat_graph_only_device"] = timed(lambda: replay(p0), n=20, do_flush=False)
    out["config0_step_ms"]["note"] = ("100 points -> 512^2, B=1, bin + splat fwd + fused L1(softor,sum) backward + fold (+ one 10k-vertex mesh "
                                      "randomised); wall clock per step over 200 steps, graph = PatternStep.capture replay next to SceneBatch.randomize")
    # ---- configs[1]: vocal-fold scene, B = 32: 18x18 grid pattern -> 500^2 sum texture + (5,5)/(3,3) blur (main.py:51-77), VocalFold
    #      (animated, V=20000, F=64) + Larynx (V=50000) randomised (examples/vocalfold_scene.py:73-77)
    g = torch.Generator().manual_seed(2)
    F, V1, V2, Bs = 64, 20000, 50000, 32
    frames = (torch.rand(F, V1, 3, generator=g) * 2 - 1).to(device)
    sc = ff.Scene(_Params(), device=device)
    vf = ff.entity.Mesh("mesh-VocalFold", frames[0], device)
    vf.add_train_animation(frames); vf.add_eval_animation(frames, max=F - 1)
    vf.scale_x(0.5, 2.0); vf.rotate_y(-0.25, 0.25)
    la = ff.entity.Mesh("mesh-Larynx", (torch.rand(V2, 3, generator=g) * 2 - 1).to(device), device)
    la.scale_x(0.8, 1.2); la.rotate_y(-0.1, 0.1)
    sc._meshes += [vf, la]
    sc.train()
    sb = sc.batch(seed=1)
    rays = ff.projection.Laser.generate_uniform_rays(0.0275, 18, 18)
    K = ff.utils.io.build_projection_matrix(60, 0.01, 1000.0)
    laser = ff.projection.Laser(ff.entity.Transformable("projector"), rays, K, 60.0, 0.01, 1000.0)
    pts01 = (laser.projectRaysToNDC()[:, 0:2] * 0.5 + 0.5).detach().contiguous()
    ptsB = pts01.unsqueeze(0).repeat(Bs, 1, 1).contiguous()

    def c1():
        sb.randomize(Bs)
        tex = R.splat_reduce(ptsB, 10.0, [500, 500], num_std_sum=None, reduce=("sum",))[0]
        run_postprocess(tex, blur=((5, 5), (3.0, 3.0)))
    ms = timed(c1)
    by = Bs * (8 * 250_000 + 8 * 250_000 + 24 * (V1 + V2))
    out["config1_vocalfold_B32"] = {"ms_per_32_samples": ms, "samples_per_s": Bs / (ms * 1e-3), "GBs": by / (ms * 1e-3) / 1e9,
                                    "frac_of_measured_peak": by / (ms * 1e-3) / 1e9 / peak,
                                    "note": "randomise two meshes (70k vertices, animated gather) + 324-point sum texture at 500^2 + 5x5 blur per sample"}
    # ---- configs[3]: post-processing, 64 x 1024^2 frames: blur (3,3) sigma (5,5) + white noise (0, 0.05) + clip
    Bf, H, W = 64, 1024, 1024
    x = torch.rand(Bf, H, W, device=device)
    gates_on = torch.ones(Bf, 2, dtype=torch.uint8, device=device)
    ms = timed(lambda: run_postprocess(x, gates=gates_on, seed=1, frame0=0, blur=((3, 3), (5.0, 5.0)), noise=(0.0, 0.05)))
    gbs = 8 * Bf * H * W / (ms * 1e-3) / 1e9
    out["config3_postprocess_64x1024x1024"] = {"ms_per_64_frames": ms, "frames_per_s": Bf / (ms * 1e-3), "GBs": gbs,
                                               "frac_of_measured_peak": gbs / peak, "note": "blur3x3 + noise + clip, both gates on, 8 B/texel"}
    return out


def main_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device: fireflies_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    # stdout carries exactly one JSON line: NCCL's own banner (NCCL_DEBUG=VERSION in this image) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    import fireflies_b200 as ff
    from fireflies_b200 import _native as nat
    from fireflies_b200 import parallel as par
    from fireflies_b200.parallel import max_over_ranks, shard_samples

    B, K, Wm = args.batch, args.steps, max(args.warmup, 3)
    hw = TS[0] * TS[1]
    first, _ = shard_samples(B * world, rank, world)

    # ---- N > 1: correctness of the exchange, of the sample split and of the sharded gradient, before anything is timed ----
    mg_check = None
    if world > 1 and os.environ.get("FFB_BENCH_SKIP_SELFCHECK") != "1":
        try:
            mg_check = par.multi_gpu_selfcheck(device)
        except AssertionError as exc:
            sys.stderr.write(f"bench.py: multi-GPU self check FAILED on rank {rank}: {exc}\n")
            os.dup2(saved_stdout, 1)
            if rank == 0:
                print(json.dumps({"metric": METRIC, "impl": "ours", "multi_gpu_check": {"failed": str(exc)}, "n_gpus": world}))
            sys.stdout.flush()
            os._exit(3)

    # ---- resident inputs ----
    g0 = torch.Generator().manual_seed(0)
    pattern = (torch.rand(N_POINTS, 2, generator=g0) * 0.96 + 0.02).to(device)
    gdev = torch.Generator(device=device).manual_seed(4 + rank)
    gS = torch.randn(B, TS[0], TS[1], device=device, generator=gdev)       # layout of baked_sum_2 ([ts0, ts1])
    gO = torch.randn(B, TS[1], TS[0], device=device, generator=gdev)
    scene = build_scene(ff, device)
    sb = scene.batch(seed=1234)
    step_obj = ff.PatternStep(N_POINTS, TS, SIGMA, B, scene_batch=sb, device=device)
    phases = ["prepare", "fwd", "bwd", "fold"]
    marks = [dict() for _ in range(K)]

    def one_step(i, rec=None):
        # the public API: randomise B scenes (side stream) | bin + splat forward -> backward against the resident upstream
        # gradients -> fold over the samples + allreduce over the ranks
        return step_obj.forward_backward(pattern, upstream=(gS, gO), sample0=i * B * world + first, marks=rec)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    for i in range(Wm):
        one_step(i)
    barrier()
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    os.close(saved_stdout)
    clocks = ClockSampler(local)
    clocks.start()
    l0 = nat.launch_count
    e0, e1 = ev(), ev()
    # like timeit: no cyclic garbage collection inside a timed region.  The host enqueues the first timed step with an empty device
    # queue behind it; a generation-2 collection there (milliseconds with torch's object graph loaded) starves the device once.
    gc.collect()
    gc.disable()
    barrier()
    e0.record()
    for i in range(K):
        _, last_dp, last_res = one_step(Wm + i, marks[i])
    e1.record()
    gc.enable()
    clocks.go()                                            # the device is K steps behind the host here: samples are under load
    barrier()
    par.check_folders()                                    # the peer-memory allreduce reports a missing peer instead of hanging
    total_ms = max_over_ranks(e0.elapsed_time(e1), device)
    launches = nat.launch_count - l0          # our kernels only (the NCCL allreduce is not counted)
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:     # before the shared-pattern and e2e runs below reuse the step's buffers
        dump_outputs(args.dump_outputs, last_dp, last_res, step_obj.last[:2])
    ms_step = total_ms / K
    value = B * world * K / (total_ms * 1e-3)
    order = ["start"] + phases[:-1] + ["end"]
    ph_ms = {p: sum(m[order[j]].elapsed_time(m[order[j + 1]]) for m in marks) / K for j, p in enumerate(phases)}
    ph_ms["randomize"] = sum(m["randomize0"].elapsed_time(m["randomize1"]) for m in marks) / K      # side stream, concurrent with prepare / fwd

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    spec = 8000.0
    alg = {"fwd": B * (8 * hw + 8 * N_POINTS), "bwd": B * (8 * hw + 16 * N_POINTS), "randomize": B * 24 * V_MESH}
    dom = max(("fwd", "bwd"), key=lambda p: ph_ms[p])
    traffic, traffic_src = None, None
    # dense patterns run the backward as splat_bwd_stp (chunks of consecutive items per CTA; FFB_SPLAT_BWD_PERSIST=0: splat_bwd_st)
    kname = {"fwd": "splat_fwd_tma", "bwd": "splat_bwd_st" if os.environ.get("FFB_SPLAT_BWD_PERSIST") == "0" else "splat_bwd_stp"}[dom]
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(tpath):                   # DRAM bytes per sample from the committed ncu --set full capture, scaled to this launch
        tj = json.load(open(tpath))
        per_sample = tj.get("per_sample_bytes", {}).get(kname)
        traffic = per_sample * B if per_sample else None
        traffic_src = tj.get("source")
    ach = alg[dom] / (ph_ms[dom] * 1e-3) / 1e9
    step_bytes = B * (16 * hw + 16 * N_POINTS + 24 * V_MESH)
    step_ach = step_bytes / (ms_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": kname, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "frac_of_spec_8TBs": ach / spec, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg[dom],
                "whole_step": {"achieved": step_ach, "frac": step_ach / peak, "frac_of_spec_8TBs": step_ach / spec,
                               "algorithmic_bytes_per_step": step_bytes},
                "kernels_ms": ph_ms,
                "kernels_gbs": {p: alg[p] / (ph_ms[p] * 1e-3) / 1e9 for p in alg},
                "kernels_frac": {p: alg[p] / (ph_ms[p] * 1e-3) / 1e9 / peak for p in alg}}

    # ---- optimisation mode, reported separately (SURVEY.md 8(d)): one pattern shared by all scenes of the step ----
    # The B textures are then one texture and the backward is linear in the upstream gradients: fold them over the samples
    # (streaming read), one forward, one backward.  NOT the headline: `value` keeps per-sample textures.
    shared = None
    if not args.no_e2e:
        step_sh = ff.PatternStep(N_POINTS, TS, SIGMA, B, scene_batch=sb, per_sample_points=False, device=device)
        for i in range(2):
            step_sh.forward_backward(pattern, upstream=(gS, gO), sample0=i * B * world + first)
        barrier()
        s0, s1 = ev(), ev()
        s0.record()
        for i in range(K):
            step_sh.forward_backward(pattern, upstream=(gS, gO), sample0=(2 + i) * B * world + first)
        s1.record()
        barrier()
        sh_ms = max_over_ranks(s0.elapsed_time(s1), device) / K
        sh_bytes = B * (8 * hw + 24 * V_MESH)                    # both upstream gradients read once + the vertex transform
        shared = {"value": B * world / (sh_ms * 1e-3), "unit": UNIT, "ms_per_step": sh_ms,
                  "achieved_GBs": sh_bytes / (sh_ms * 1e-3) / 1e9, "frac_of_peak": sh_bytes / (sh_ms * 1e-3) / 1e9 / peak,
                  "note": "PatternStep(per_sample_points=False): upstream gradients folded over the samples, one forward + one backward; "
                          "a separate mode, not the headline metric"}
        del step_sh

    # ---- e2e: public API with host buffers ----
    e2e = None
    if not args.no_e2e:
        pts_host = pattern.cpu().pin_memory()
        out_host = torch.empty(N_POINTS, 2).pin_memory()
        loss_host = torch.empty(B).pin_memory()
        del gS, gO
        torch.cuda.empty_cache()
        for i in range(2):
            step_obj.step_host(pts_host, out_host, loss_host, sample0=i * B * world + first)
        gc.collect()
        gc.disable()
        barrier()
        t0 = time.perf_counter()
        for i in range(K):
            step_obj.step_host(pts_host, out_host, loss_host, sample0=(2 + i) * B * world + first)
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0, device)
        gc.enable()
        e2e = {"value": B * world * K / dt, "unit": UNIT, "h2d_bytes_per_step": pts_host.numel() * 4,
               "d2h_bytes_per_step": (out_host.numel() + loss_host.numel()) * 4, "ms_per_step": dt / K * 1e3,
               "path": "PatternStep.step_host: pinned pattern H2D -> randomise (side stream) | bin + splat fwd -> fused L1(softor,sum) "
                       "loss + backward (rasterization.py:589-599, ffb_splat_bwd_l1) -> fold -> allreduce -> gradient+loss D2H"}

    side = None
    if rank == 0 and world == 1 and not args.no_side:
        try:
            side = side_configs(ff, device, peak)
        except Exception as exc:  # noqa: BLE001  (a side measurement must not take the headline line down)
            side = {"error": repr(exc)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n = 40                                                    # ~12 s of CPU work on the box (3.4 samples/s)
        v, cores, dt = run_cpu(n)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{n} scene samples of the 256-scene step at full size ({dt:.1f} s of CPU work), linear extrapolation"}

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config(B, world), "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "shared_pattern_mode": shared,
            "multi_gpu_check": mg_check, "side": side, "gpu_launches": launches,
            "clocks": clk}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        main_reference(a)
    else:
        main_ours(a)
