"""Times the transform backward on the GPU (CUDA events around CUDA-graph replays, so host launch cost stays out):

  points   ffb_transform_points_bwd            d_pts only        24 B read + 12 B written per point
  full     ffb_transform_points_bwd_full       d_pts + d_T       24 B read + 12 B written per point
  dT       ffb_transform_points_bwd_full       d_T only          24 B read per point

at V = 1e5, 1e6 and 1e7 points (the last one's 360 MB working set exceeds the 126 MB L2; the smaller ones are read from L2
after the first pass).  Each size is warmed up, then the variants alternate in blocks of 10 launches until every variant has
run at least --launches launches.  Before timing, the outputs are checked: d_pts of the fused entry equals the points-only
kernel's bit for bit, and d_T is within 1e-5 of the fp64 closed form per entry (relative to the sum of |terms|).  Prints one
JSON line with the card name and power limit read in the same run; --out also writes it to a file.

    python scripts/transform_grad_time.py [--launches 200] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BLOCK = 10
BYTES = {"points": 36, "full": 36, "dT": 24}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unavailable ({e})"
    return name, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--sizes", type=str, default="100000,1000000,10000000")
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("transform_grad_time.py needs a CUDA device")
    from fireflies_b200 import _native as nat
    L = nat.lib()
    name, power = card()
    rows = []
    gen = torch.Generator(device="cuda").manual_seed(0)
    for V in [int(v) for v in a.sizes.split(",")]:
        pts = torch.randn((V, 3), device="cuda", generator=gen)
        pts[:, 2] = -1.0 - 4.0 * torch.rand(V, device="cuda", generator=gen)
        g = torch.randn((V, 3), device="cuda", generator=gen)
        T = torch.tensor([[1.7320509, 0, 0, 0], [0, 1.7320509, 0, 0], [0, 0, -1.00001, -0.0100001], [0, 0, -1, 0]],
                         device="cuda")
        d_a, d_b = torch.empty_like(pts), torch.empty_like(pts)
        dT = torch.empty(16, device="cuda")
        nb = L.ffb_transform_bwd_workspace_bytes(V)
        ws = torch.empty(max(nb, 1), dtype=torch.uint8, device="cuda")
        wsp = ws.data_ptr() if nb else None

        def launch(kind):
            s = torch.cuda.current_stream().cuda_stream
            if kind == "points":
                rc = L.ffb_transform_points_bwd(pts.data_ptr(), V, T.data_ptr(), 0, g.data_ptr(), d_a.data_ptr(), s)
            else:
                rc = L.ffb_transform_points_bwd_full(pts.data_ptr(), V, T.data_ptr(), 0, g.data_ptr(),
                                                     d_b.data_ptr() if kind == "full" else None, dT.data_ptr(), wsp, nb, s)
            assert rc == 0, L.ffb_last_error_string()

        for k in BYTES:
            launch(k)
        torch.cuda.synchronize()
        assert torch.equal(d_a, d_b), "fused d_pts differs from the points-only kernel"
        p64, g64, T64 = pts.double().cpu().numpy(), g.double().cpu().numpy(), T.double().cpu().numpy()
        pt = np.hstack([p64, np.ones((V, 1))])
        h = pt @ T64.T
        inv = 1.0 / h[:, 3]
        d = np.hstack([g64 * inv[:, None], (-(g64 * h[:, :3]).sum(1) * inv * inv)[:, None]])
        ref, scale = d.T @ pt, np.abs(d).T @ np.abs(pt)
        err = float((np.abs(dT.view(4, 4).cpu().numpy() - ref) / np.maximum(scale, 1e-300)).max())
        assert err <= 1e-5, err

        graphs = {}
        for k in BYTES:
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                for _ in range(BLOCK):
                    launch(k)
            graphs[k] = gr
        for _ in range(3):                                     # warm-up
            for k in BYTES:
                graphs[k].replay()
        torch.cuda.synchronize()
        ms = {k: 0.0 for k in BYTES}
        rounds = -(-a.launches // BLOCK)
        order = list(BYTES)
        for r in range(rounds):
            for k in order[r % 3:] + order[:r % 3]:            # rotate which variant goes first
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                graphs[k].replay()
                e1.record()
                e1.synchronize()
                ms[k] += e0.elapsed_time(e1)
        n = rounds * BLOCK
        row = {"V": V, "working_set_MB": round(V * 36 / 1e6, 1), "launches": n, "dT_err_rel_sum_abs": err}
        for k in BYTES:
            t = ms[k] / n
            row[f"{k}_ms"] = round(t, 5)
            row[f"{k}_GBps"] = round(V * BYTES[k] / (t * 1e-3) / 1e9, 1)
        row["full_over_points"] = round(row["full_ms"] / row["points_ms"], 3)
        rows.append(row)
        del graphs
    res = {"device": name, "power_limit_and_max_sm_clock": power, "rows": rows}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
