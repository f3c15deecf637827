"""Batched rendering (AmbientOcclusion.render_batch, one context, one stream, one graph replay per batch) against the two
single-frame ways of pushing the same frames through a B200, in ONE process:

  batch   render_batch of B frames on one stream (B = 1 / 4 / 16 / 64 at 1920x1080, B = 8 at 3840x2160);
  replica the same frames round-robin over 5 contexts on 5 streams (bench.py's throughput method);
  serial  one frame after the other through one context on one stream.

Frames are distinct (generated with bench.make_depth and shifted), and a batch's inputs plus intermediates exceed the
126 MB L2.  Each arm is warmed up, then timed with CUDA events over >= 5 windows of >= 0.2 s; the median window gives
us/frame and Mpx/s.  Every frame of the timed 64-frame batch (and of the 4K batch) is checked against single-frame render.

    python scripts/bench_batch.py --out profiles/r3_batch_b200.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (make_depth; bench.py guards its __main__)

WINDOWS, MIN_WINDOW_S, N_REPLICAS = 7, 0.2, 5


def gpu_info() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:      # noqa: BLE001 -- the numbers still stand, the label says it is missing
        return {"name": "unknown", "error": str(e)}


def timed(torch, submit, streams, per_window_hint: int) -> tuple[float, int]:
    """Median ms of one submit() over WINDOWS windows of >= MIN_WINDOW_S each (CUDA events on every stream)."""
    def window(n):
        # one start event that every stream waits for, one end event after every stream's last kernel
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(streams[0])
        for s in streams[1:]:
            s.wait_event(start)
        for i in range(n):
            submit(i)
        for s in streams[1:]:
            e = torch.cuda.Event()
            e.record(s)
            streams[0].wait_event(e)
        end.record(streams[0])
        torch.cuda.synchronize()
        return start.elapsed_time(end)
    n = max(1, per_window_hint)
    while True:
        ms = window(n)
        if ms >= MIN_WINDOW_S * 1e3:
            break
        n = int(n * max(2.0, 1.2 * MIN_WINDOW_S * 1e3 / max(ms, 1e-3))) + 1
    per = [window(n) / n for _ in range(WINDOWS)]
    return statistics.median(per), n


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sweep", default="1,4,16,64")
    args = ap.parse_args()
    import numpy as np
    import torch
    from miniengineao_b200 import AmbientOcclusion, Camera
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "windows": WINDOWS, "min_window_s": MIN_WINDOW_S, "replicas": N_REPLICAS, "rows": []}

    def frames(W, H, n):
        host = [torch.from_numpy(bench.make_depth(W, H, f)) for f in range(4)]
        return torch.stack([torch.roll(host[i % 4], shifts=29 * (i // 4), dims=1) for i in range(n)]).to(dev).contiguous()

    def ctx(W, H):
        ao = AmbientOcclusion(Camera(W, H), device=0)
        ao.intensity = bench.INTENSITY
        return ao

    def run(W, H, B, check):
        depth = frames(W, H, B)
        out = torch.empty((B, H, W), dtype=torch.uint8, device=dev)
        mpx = W * H / 1e6
        row = {"W": W, "H": H, "B": B}
        # batch: one context, one stream
        a = ctx(W, H)
        a.reserve_batch(B)
        s = torch.cuda.Stream(device=dev)
        for _ in range(3):
            a.render_batch(depth, out, stream=s)
        torch.cuda.synchronize()
        ms, n = timed(torch, lambda i: a.render_batch(depth, out, stream=s), [s], 4)
        row["batch_us_per_frame"] = 1e3 * ms / B
        row["batch_mpx_s"] = mpx * B / ms * 1e3
        # replicas: the same frames over 5 contexts / streams
        ctxs = [ctx(W, H) for _ in range(N_REPLICAS)]
        sts = [torch.cuda.Stream(device=dev) for _ in range(N_REPLICAS)]
        rep_out = torch.empty_like(out)

        def rsub(i):
            for f in range(B):
                k = (i * B + f) % N_REPLICAS
                ctxs[k].render(depth[f], rep_out[f], stream=sts[k])
        for i in range(2):
            rsub(i)
        torch.cuda.synchronize()
        ms_r, _ = timed(torch, rsub, sts, 4)
        row["replica_us_per_frame"] = 1e3 * ms_r / B
        row["replica_mpx_s"] = mpx * B / ms_r * 1e3
        # serial: one context, one stream, one frame after the other
        c1, s1 = ctxs[0], sts[0]

        def ssub(i):
            for f in range(B):
                c1.render(depth[f], rep_out[f], stream=s1)
        ssub(0)
        torch.cuda.synchronize()
        ms_s, _ = timed(torch, ssub, [s1], 4)
        row["serial_us_per_frame"] = 1e3 * ms_s / B
        row["serial_mpx_s"] = mpx * B / ms_s * 1e3
        row["batch_vs_serial"] = ms_s / ms
        row["batch_vs_replica"] = ms_r / ms
        if check:       # every frame of the timed batch equals its single-frame render
            a.render_batch(depth, out, stream=s)
            torch.cuda.synchronize()
            single = torch.empty_like(out)
            for f in range(B):
                c1.render(depth[f], single[f], stream=s1)
            torch.cuda.synchronize()
            row["frames_differing_from_render"] = int((out != single).flatten(1).any(1).sum().item())
        print(json.dumps(row), flush=True)
        res["rows"].append(row)
        del a, ctxs
        torch.cuda.synchronize()

    for B in [int(x) for x in args.sweep.split(",")]:
        run(1920, 1080, B, check=(B == 64))
    run(3840, 2160, 8, check=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
