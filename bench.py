#!/usr/bin/env python
"""bench.py -- Mpixels/s of the full multi-scale SSAO pipe (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload 4k|1080p|8k|256] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" = one frame through the whole hot path (prepare_depth, 4x render_ao, 4x blur_upsample).
Headline (every N): the 3840x2160 frame the metric is quoted on (BASELINE.json configs[2]); at N > 1 every rank renders its own
frames -- weak scaling, no data-path collective (the reference keeps no temporal state, frames are independent).

  value     device-resident throughput: R batches of EXACTLY K graph replays, each batch bracketed by barrier + synchronize, timed
            with CUDA events, max over ranks; the MEDIAN batch is reported (all batches listed).  Each step reads a different one
            of 8 depth frames (8 x 33 MB > the 126 MB L2), so inputs are HBM-cold
  e2e       the same metric through AmbientOcclusion.render_host_batch (C ABI meao_render_host_async / meao_host_wait): pinned
            HOST depth in, HOST AO out, H2D + nine kernels + D2H inside the timed region of every step; f32 depth (what the
            reference arm consumes) is the e2e value, native D16 ingest is reported beside it
  roofline  dominant kernel: algorithmic bytes of the reference data-flow (SURVEY.md 8d) / its mean device time (CUDA events
            around every kernel, same process) vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the CPU oracle (scalar C restatement of the reference compute shaders) on this host
  configs   the other BASELINE.json configs, each with its own number: 256^2 single-scale (configs[0]), 1080p (configs[1]),
            8K single frame -- on one GPU at N = 1, row-banded over the N GPUs with the native NVLink halo exchange at N > 1
            (configs[3]; speed-up against the one-GPU 8K time measured in the same run), batch of 64 x 1080p (configs[4])
--impl reference: times that CPU restatement alone (the reference itself is HLSL + Unity C#, which cannot be built or run in
this image: see DESIGN.md), all host threads, same workload / metric / config string.
--dump-outputs DIR: after the timed steps, DIR/ao.npy (float32) holds the AO codes of the headline's last timed step (rank 0;
            --impl reference: the oracle's last timed frame).  Inputs are generated deterministically, so two builds run with the
            same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

# several contexts per GPU handshake through spinning exchange kernels in the band mode: one hardware queue per stream
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {"256": (256, 256), "1080p": (1920, 1080), "4k": (3840, 2160), "8k": (7680, 4320)}
METRIC = "Mpixels/sec full SSAO pipe @4K"
INTENSITY = 1.1   # Sponza.unity:969; every other parameter at the component default (AO.cs:20-52)
BATCHES = 5       # timed batches of K steps; the median is the headline
DUMP_BYTES = 64_000_000   # --dump-outputs budget


def dump_output(dir_: str, name: str, a: np.ndarray) -> None:
    """DIR/<name>.npy in float32.  An array above DUMP_BYTES is cut to a fixed sample of its flattened elements (the sorted
    positions np.random.default_rng(0) picks), so dumps of the same workload still compare element for element."""
    a = np.asarray(a, dtype=np.float32)
    cap = DUMP_BYTES // 4 - 1024          # room for the .npy header
    if a.size > cap:
        a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
    os.makedirs(dir_, exist_ok=True)
    np.save(os.path.join(dir_, f"{name}.npy"), a)


def workload_label(W: int, H: int) -> str:
    """The config.workload string -- identical in both arms."""
    return f"{W}x{H} synthetic Sponza-like corridor depth, full multi-scale pipe, component defaults, intensity {INTENSITY}"


def load_peaks() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def pin_to_gpu_numa(local: int) -> dict:
    """Bind this process (and the pinned buffers it allocates afterwards) to the CPUs of the GPU's NUMA node."""
    info = {"numa_node": None, "cpus": None}
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return info
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info = {"numa_node": node, "cpus": len(allowed)}
    except Exception as e:      # not fatal: the run is merely unpinned
        info["error"] = str(e)[:80]
    return info


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def make_depth(W: int, H: int, frame: int, row0: int = 0, row1: int | None = None) -> np.ndarray:
    from miniengineao_b200 import synth
    return synth.lin01_to_raw(synth.corridor(W, H, frame=frame, row0=row0, row1=row1))


def cpu_oracle_run(W: int, H: int, depth: np.ndarray, threads: int, reps: int, **kw) -> float:
    """Mpixels/s of the CPU oracle (kind = "port") -- the checker, timed as the CPU baseline."""
    from oracle.oracle import Oracle
    o = Oracle(W, H, threads=threads, intensity=INTENSITY, **kw)
    o.run(depth)                       # warm-up (page faults, caches, worker pool)
    ts = []
    for _ in range(reps):
        t = time.perf_counter(); o.run(depth); ts.append(time.perf_counter() - t)
    return W * H / statistics.median(ts) / 1e6


def pick_cpu_threads(W: int, H: int, depth: np.ndarray) -> int:
    """All logical CPUs or one thread per physical core, whichever is faster here (SMT siblings often lose on this FP-dense code)."""
    from oracle.oracle import Oracle
    cores = os.cpu_count() or 1
    cands = sorted({cores, max(1, cores // 2)}, reverse=True)
    best, best_t = cands[0], float("inf")
    for c in cands:
        o = Oracle(W, H, threads=c, intensity=INTENSITY)
        o.run(depth)
        ts = []
        for _ in range(3):
            t = time.perf_counter(); o.run(depth); ts.append(time.perf_counter() - t)
        if statistics.median(ts) < best_t:
            best, best_t = c, statistics.median(ts)
    return best


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    W, H = WORKLOADS[args.workload]
    depth = make_depth(W, H, 0)
    from oracle.oracle import Oracle
    cores = pick_cpu_threads(W, H, depth)
    o = Oracle(W, H, threads=cores, intensity=INTENSITY)
    # each step = one frame (the same single frame every step); exactly K timed steps
    steps, warm = args.steps, max(0, min(args.warmup, 32))
    for _ in range(warm):
        o.run(depth)
    t0 = time.perf_counter()
    for _ in range(steps):
        last = o.run(depth)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_output(args.dump_outputs, "ao", last)
    v = W * H * steps / dt / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "Mpixels/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": workload_label(W, H),
                                             "note": "CPU restatement of the reference compute shaders (oracle/meao_oracle.c), persistent worker pool; "
                                                     "the reference itself is HLSL + Unity C# and cannot run here"},
            "cpu_baseline": {"value": v, "unit": "Mpixels/s", "cores": cores, "kind": "port",
                             "sample": f"{steps} x one {W}x{H} frame, {cores} pooled pthreads over (thread-group row x column range) units; "
                                       f"thread count picked from {{{os.cpu_count()}, {max(1, (os.cpu_count() or 1) // 2)}}} by a 3-frame trial"},
            "e2e": {"value": v, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_ours(args) -> None:
    import torch
    import torch.distributed as dist
    from miniengineao_b200 import AmbientOcclusion, Camera

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (there is no CPU fallback); use --impl reference for the CPU arm")
    numa = pin_to_gpu_numa(local)           # before any pinned allocation: first-touch places the staging buffers on the GPU's node
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    W, H = WORKLOADS[args.workload]
    K, Wm = args.steps, max(args.warmup, 3)
    NBUF = 8
    S = max(1, args.streams)
    BAND_ONLY = args.only_8k

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def mk_contexts(w, h, n, **attrs):
        out = []
        for _ in range(n):
            a_ = AmbientOcclusion(Camera(w, h), device=local)
            a_.intensity = INTENSITY
            for k_, v_ in attrs.items():
                setattr(a_, k_, v_)
            out.append(a_)
        return out

    def timed_batches(submit, streams, k, batches=BATCHES) -> list[float]:
        """`batches` timed regions of EXACTLY k submit() calls, each bracketed by barrier + synchronize; device time (CUDA
        events on the stream that forks to / joins from the worker streams), max over ranks."""
        main = torch.cuda.current_stream(dev)
        out = []
        for _ in range(batches):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record(main)
            for st in streams:
                st.wait_event(e0)
            for i in range(k):
                submit(i)
            for st in streams:
                ev = torch.cuda.Event()
                ev.record(st)
                main.wait_event(ev)
            e1.record(main)
            barrier()
            out.append(allmax(e0.elapsed_time(e1)))
        return out

    def throughput(w, h, depths, outs, k, n_ctx=S, **attrs):
        """Frame stream over n_ctx contexts / streams (frames are independent).  Returns (median ms per batch, batches, contexts)."""
        ctxs = mk_contexts(w, h, n_ctx, **attrs)
        sts = [torch.cuda.Stream(device=dev) for _ in range(n_ctx)]
        nb = len(depths)

        def submit(i):
            ctxs[i % n_ctx].render(depths[i % nb], outs[i % len(outs)], stream=sts[i % n_ctx])
        for i in range(max(nb, n_ctx) * n_ctx):        # set-up: captures one graph per (context, buffer pair) the stream will use
            submit(i)
        torch.cuda.synchronize()
        for i in range(Wm):
            submit(i)
        ms = timed_batches(submit, sts, k)
        return statistics.median(ms), ms, ctxs, sts, submit

    if BAND_ONLY:       # development aid: just the row-banded 8K measurement (not a bench line the driver uses)
        peak, _ = load_peaks()
        r = bench_8k(args, torch, dist if world > 1 else None, dev, rank, world, local, barrier, allmax, timed_batches, mk_contexts, peak)
        if rank == 0:
            print(json.dumps(r), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ================= headline: 4K (or --workload) frames, device resident =================================================
    frames_host = [make_depth(W, H, f + 64 * rank) for f in range(2)]
    depths = []
    for i in range(NBUF):       # 8 distinct device frames (2 generated + shifted copies: content differs, cost of generation bounded)
        base = torch.from_numpy(frames_host[i % 2]).to(dev)
        depths.append(torch.roll(base, shifts=37 * (i // 2), dims=1).contiguous() if i >= 2 else base)
    outs = [torch.empty((H, W), dtype=torch.uint8, device=dev) for _ in range(NBUF)]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    ms_med, ms_batches, aos, streams, submit = throughput(W, H, depths, outs, K)
    # the last timed step wrote outs[(K - 1) % NBUF] (earlier steps on that buffer read the same depth frame)
    last_ao = outs[(K - 1) % NBUF].cpu().numpy() if args.dump_outputs and rank == 0 else None
    ao = aos[0]
    launches = K * ao.kernels_per_frame
    t_end = time.time() + 0.6               # keep the load up a little longer so the 100 ms clock sampler sees it
    while time.time() < t_end:
        for i in range(64):
            submit(i)
        torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    value = W * H * K * world / (ms_med * 1e-3) / 1e6

    # the same K frames strictly one after the other on ONE stream / context (what a single camera sees: latency)
    def serial_ms(ctx, dl, ol, k):
        ts = []
        for _ in range(3):
            torch.cuda.synchronize()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for i in range(k):
                ctx.render(dl[i % len(dl)], ol[i % len(ol)])
            s1.record()
            torch.cuda.synchronize()
            ts.append(s0.elapsed_time(s1) / k)
        return statistics.median(ts)
    ms_serial = serial_ms(ao, depths, outs, K)

    # ================= end to end through the host-buffer API ==================================================================
    import ctypes as C
    from miniengineao_b200 import _native as N
    lib = N.lib()
    hps = [lib.meao_host_alloc(W * H * 4) for _ in range(2)]
    ops = [lib.meao_host_alloc(W * H) for _ in range(2)]
    hds = [np.ctypeslib.as_array(C.cast(p_, C.POINTER(C.c_float)), shape=(H, W)) for p_ in hps]
    h16 = [np.ctypeslib.as_array(C.cast(p_, C.POINTER(C.c_uint16)), shape=(H, W)) for p_ in hps]      # the same pinned memory, D16 view
    hos = [np.ctypeslib.as_array(C.cast(p_, C.POINTER(C.c_uint8)), shape=(H, W)) for p_ in ops]
    Ke = max(8, min(K, 60))

    def e2e_run(bufs):
        ao.render_host_batch([bufs[i & 1] for i in range(4)], [hos[i & 1] for i in range(4)])        # warm-up
        barrier()
        t0 = time.perf_counter()
        # every step: H2D of that step's depth from pinned host memory, the nine kernels, D2H of its AO texture;
        # render_host_batch alternates two staging slots so the copies of neighbouring steps overlap the kernels
        ao.render_host_batch([bufs[i & 1] for i in range(Ke)], [hos[i & 1] for i in range(Ke)])
        torch.cuda.synchronize()
        return W * H * Ke * world / allmax(time.perf_counter() - t0) / 1e6
    for i in range(2):
        hds[i][...] = frames_host[i]
    e2e_value = e2e_run(hds)
    t0 = time.perf_counter()                # the strictly serial form (one blocking call per frame) for comparison
    for i in range(10):
        ao.render_host(hds[i & 1], hos[i & 1])
    e2e_serial = W * H * 10 / (time.perf_counter() - t0) / 1e6
    ao.render_host(hds[0], hos[0])
    ho = hos[0].copy()
    e2e_check = int(ho.astype(np.uint64).sum())
    # native D16 ingest (MEAO_DEPTH_RAW_D16_UNORM, what a D16 camera target would hand over): half the upload
    for i in range(2):
        h16[i][...] = np.clip(np.rint(frames_host[i].astype(np.float64) * 65535.0), 1, 65535).astype(np.uint16)
    e2e_d16 = e2e_run(h16)

    # ================= per-kernel device times (events around every kernel), rank 0 ===========================================
    roofline, kernels = None, None
    if rank == 0:
        peak, peak_src = load_peaks()
        acc: dict[str, list[float]] = {}
        PREP = 8        # launches per kernel inside one event pair: the pair's overhead and the launch gap are amortised (kernels are idempotent)
        for i in range(12):
            for name, kms in ao.profile_frame(depths[i % NBUF], outs[i % NBUF], repeats=PREP):
                acc.setdefault(name, []).append(kms)
        means = {k: statistics.mean(v[2:]) for k, v in acc.items()}
        acc1: dict[str, list[float]] = {}
        for i in range(6):      # and single launches (what round 1 reported: includes ~2-3 us of launch gap per kernel)
            for name, kms in ao.profile_frame(depths[i % NBUF], outs[i % NBUF], repeats=1):
                acc1.setdefault(name, []).append(kms)
        single = {k: statistics.mean(v[2:]) for k, v in acc1.items()}
        px = lambda l: ((W + (1 << l) - 1) >> l) * ((H + (1 << l) - 1) >> l)  # noqa: E731
        alg = {"prepare_depth": ao.algorithmic_bytes(1) + ao.algorithmic_bytes(2)}
        for k in range(1, 5):
            alg[f"render_ao L{k}"] = 32 * px(k + 2) + px(k)
        for lo in range(4, 0, -1):
            hi = lo - 1
            alg[f"blur_upsample L{lo}->L{hi}"] = 5 * px(lo) + (2 if hi == 0 else 5) * px(hi) + px(hi)
        kernels = {k: {"ms": round(means[k], 5), "ms_single_launch": round(single[k], 5), "alg_bytes": alg[k],
                       "alg_gbs": round(alg[k] / (means[k] * 1e-3) / 1e9, 1)} for k in means}
        dom = max(means, key=lambda k: means[k])
        ach = alg[dom] / (means[dom] * 1e-3) / 1e9
        total_alg = ao.algorithmic_bytes(0)
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic_4k.json")) as f:
                tj = json.load(f)
            if tj.get("workload") == f"{W}x{H}":
                traffic = tj["dram_bytes_per_launch"].get(dom)
                traffic_src = f"profiles/traffic_4k.json ({tj.get('build', 'ncu dram__bytes_read+write of that kernel, one cold launch')})"
        except Exception:
            pass
        roofline = {"bound": "hbm", "kernel": dom, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                    "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peak_src, "algorithmic_bytes": alg[dom],
                    "timing": f"mean device time of that kernel over {PREP} back-to-back launches inside one CUDA-event pair, 10 frames (single launches: "
                              f"{single[dom] * 1e3:.1f} us incl. the launch gap); inputs L2-resident as in the pipeline",
                    "note": "the kernel is instruction-issue bound, not HBM bound (bit-exact IEEE divisions; see DESIGN.md 5)",
                    "pipe_algorithmic_bytes": total_alg,
                    "pipe_achieved": round(total_alg * K / (ms_med * 1e-3) / 1e9, 1),
                    "pipe_frac": round(total_alg * K / (ms_med * 1e-3) / 1e9 / peak, 4),
                    "kernel_share_of_step": round(means[dom] / sum(means.values()), 4)}

    # ================= the consumer end (SURVEY.md 8f.1): frame-buffer composite, a genuinely HBM-bound kernel ================
    composite = None
    if rank == 0 and not args.quick:
        peak, _ = load_peaks()
        comp = {}
        for name, dt_, bpp in (("rgba16f", torch.float16, 8), ("rgba8", torch.uint8, 4)):
            bufs = [torch.zeros((H, W, 4), dtype=dt_, device=dev) for _ in range(6)]     # 6 x 66 MB > L2 for rgba16f
            for b_ in bufs:
                ao.composite_framebuffer(outs[0], b_)
            torch.cuda.synchronize()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 30
            c0.record()
            for i in range(reps):
                ao.composite_framebuffer(outs[i % NBUF], bufs[i % 6])
            c1.record()
            torch.cuda.synchronize()
            us = c0.elapsed_time(c1) / reps * 1e3
            nbytes = W * H * (2 * bpp + 1)
            comp[name] = {"us": round(us, 2), "bytes": nbytes, "gbs": round(nbytes / us / 1e3, 1), "frac_of_peak": round(nbytes / us / 1e3 / peak, 3)}
            del bufs
        composite = {"kernel": "composite_framebuffer (Blit.shader pass 2: colour *= ao), read + write colour + read ao", **comp}

    # ================= CPU baseline beside it (rank 0, N = 1 only) =============================================================
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            os.sched_setaffinity(0, range(os.cpu_count() or 1))       # the CPU arm gets every core, not just the GPU's NUMA node
        except OSError:
            pass
        cores = pick_cpu_threads(W, H, frames_host[0])
        v_all = cpu_oracle_run(W, H, frames_host[0], cores, 5)
        v_one = cpu_oracle_run(W, H, frames_host[0], 1, 2)
        cpu = {"value": round(v_all, 2), "unit": "Mpixels/s", "cores": cores, "kind": "port",
               "sample": f"5 x one {W}x{H} frame, median, {cores} pooled pthreads over (thread-group row x column range) units "
                         f"(of {os.cpu_count()} logical CPUs; count picked by a 3-frame trial); value_1thread = 2 frames on 1 thread",
               "value_1thread": round(v_one, 2)}
        from oracle.oracle import Oracle                # and the oracle agrees with what the GPU produced for that frame
        ref = Oracle(W, H, threads=cores, intensity=INTENSITY).run(frames_host[0])
        cpu["gpu_matches_oracle"] = bool(int(ref.astype(np.uint64).sum()) == e2e_check and np.array_equal(ref, ho))
        pin_to_gpu_numa(local)
    for p_ in hps + ops:
        lib.meao_host_free(p_)
    del depths, outs, aos
    torch.cuda.empty_cache()

    # ================= the other BASELINE.json configs =======================================================================
    configs = {}
    peak, _ = load_peaks()
    if not args.quick:
        # ---- configs[3]: ONE 7680x4320 frame.  N = 1: the whole frame on this GPU.  N > 1: row bands, native halo exchange ----
        configs["8k_single_frame"] = bench_8k(args, torch, dist if world > 1 else None, dev, rank, world, local, barrier, allmax,
                                             timed_batches, mk_contexts, peak)
        # ---- configs[4]: batch of 64 x 1080p, 64 / N frames per GPU, no communication ------------------------------------------
        configs["batch_64x1080p"] = bench_batch1080p(torch, dev, rank, world, throughput, peak, K)
        if rank == 0 and world == 1:
            # ---- configs[1]: 1920x1080, one GPU --------------------------------------------------------------------------------
            configs["1080p"] = bench_1080p(torch, dev, throughput, serial_ms, peak, K)
            # ---- configs[0]: 256x256 flat + sphere, single-scale plan; GPU beside the scalar CPU twin ---------------------------
            configs["256_single_scale"] = bench_256_single_scale(torch, dev, local, args)

    if rank == 0:
        line = {"metric": METRIC, "value": round(value, 1), "unit": "Mpixels/s", "n_gpus": world, "steps": K, "warmup": Wm,
                "ms_per_step": round(ms_med / K, 5), "batches_ms_per_step": [round(m / K, 5) for m in ms_batches],
                "serial_frames": {"value": round(W * H / (ms_serial * 1e-3) / 1e6, 1), "unit": "Mpixels/s",
                                  "ms_per_frame": round(ms_serial, 5), "note": "rank 0, ONE stream / context, frames back to back (single-camera latency)"},
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_label(W, H),
                           "per_gpu": "one frame per step on every rank (frames are independent; no data-path collective)",
                           "streams": f"{S} contexts on {S} CUDA streams, frames alternate (throughput mode; serial_frames = one stream)",
                           "l2": f"inputs rotate over {NBUF} distinct depth frames ({NBUF * W * H * 4 / 1e6:.0f} MB > 126 MB L2); intermediates stay L2-resident by design",
                           "timing": f"median of {BATCHES} batches of exactly {K} steps, each bracketed by barrier + synchronize, CUDA events, max over ranks; "
                                     f"{Wm} warm-up steps after the graph-capture set-up pass",
                           "pdl_level": ao.pdl_level, "numa": numa},
                "e2e": {"value": round(e2e_value, 1), "unit": "Mpixels/s", "h2d_bytes_per_step": W * H * 4, "d2h_bytes_per_step": W * H, "steps": Ke,
                        "api": "AmbientOcclusion.render_host_batch -> meao_render_host_async / meao_host_wait (pinned host buffers, 2 staging slots)",
                        "serial_value": round(e2e_serial, 1),
                        "d16_ingest": {"value": round(e2e_d16, 1), "h2d_bytes_per_step": W * H * 2, "note": "MEAO_DEPTH_RAW_D16_UNORM: the depth texture uploaded in its native 16-bit format"}},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu,
                "configs": configs, "rowtile": configs.get("8k_single_frame") if world > 1 else None, "composite": composite}
        if last_ao is not None:
            dump_output(args.dump_outputs, "ao", last_ao)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def bench_8k(args, torch, dist, dev, rank, world, local, barrier, allmax, timed_batches, mk_contexts, peak) -> dict | None:
    from miniengineao_b200 import Camera, rowtile as RT
    RW, RH = WORKLOADS["8k"]
    RS = max(1, args.band_streams)
    Kr = max(args.steps, 100)
    px = RW * RH
    alg = None

    def one_gpu(full_dev):
        """the whole 8K frame on ONE GPU, frame stream over RS contexts (the N = 1 point of the row-tile curve)."""
        ctxs = mk_contexts(RW, RH, RS)
        sts = [torch.cuda.Stream(device=dev) for _ in range(RS)]
        outs = [torch.empty((RH, RW), dtype=torch.uint8, device=dev) for _ in range(RS)]

        def sub(i):
            ctxs[i % RS].render(full_dev, outs[i % RS], stream=sts[i % RS])
        for i in range(2 * RS + 3):
            sub(i)
        torch.cuda.synchronize()
        ts = []
        for _ in range(BATCHES):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            main = torch.cuda.current_stream(dev)
            torch.cuda.synchronize()
            e0.record(main)
            for st in sts:
                st.wait_event(e0)
            for i in range(Kr):
                sub(i)
            for st in sts:
                ev = torch.cuda.Event(); ev.record(st); main.wait_event(ev)
            e1.record(main)
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / Kr)
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(40):
            ctxs[0].render(full_dev, outs[0])
        s1.record()
        torch.cuda.synchronize()
        a_bytes = ctxs[0].algorithmic_bytes(0)
        res = (statistics.median(ts), s0.elapsed_time(s1) / 40, a_bytes, outs[0].clone())
        del ctxs, outs
        return res

    if world == 1:
        full = torch.from_numpy(make_depth(RW, RH, 0)).to(dev)
        ms1, ms1_serial, alg, got = one_gpu(full)
        ok = None
        if not args.no_cpu:
            from oracle.oracle import Oracle
            ref = Oracle(RW, RH, threads=os.cpu_count() or 1, intensity=INTENSITY).run(full.cpu().numpy())
            ok = bool(np.array_equal(ref, got.cpu().numpy()))
        del full
        torch.cuda.empty_cache()
        return {"workload": f"{RW}x{RH} single frame on ONE GPU ({RS} contexts / streams; the N = 1 point of the row-tile curve)",
                "value": round(px / (ms1 * 1e-3) / 1e6, 1), "unit": "Mpixels/s", "ms_per_frame": round(ms1, 5), "steps": Kr, "batches": BATCHES,
                "serial_ms_per_frame": round(ms1_serial, 5), "roofline_frac": round(alg / (ms1 * 1e-3) / 1e9 / peak, 4),
                "matches_oracle": ok, "scaling": "strong", "n_gpus": 1}

    # ---- N > 1: contiguous 16-row-aligned bands, one per rank; RS band contexts per rank alternate over RS streams so that the
    #      halo exchange of frame i overlaps the kernels of frame i+1 (every context owns its intermediates and flags)
    mode = args.band_mode
    try:
        rts = [RT.RowTiledAO(Camera(RW, RH), rank, world, local, mode=mode, intensity=INTENSITY) for _ in range(RS)]
    except Exception as e:      # peer mappings unavailable (no P2P / IPC in this container): fall back to NCCL send/recv between two graphs
        if mode != "native":
            raise
        mode = f"p2p (native refused: {str(e)[:100]})"
        rts = [RT.RowTiledAO(Camera(RW, RH), rank, world, local, mode="p2p", intensity=INTENSITY) for _ in range(RS)]
    rt = rts[0]
    rstreams = [torch.cuda.Stream(device=dev) for _ in range(RS)]
    band = torch.from_numpy(make_depth(RW, RH, 0, rt.row0, rt.row1)).to(dev)
    obands = [torch.empty((rt.rows, RW), dtype=torch.uint8, device=dev) for _ in range(RS)]

    def rstep(i):
        with torch.cuda.stream(rstreams[i % RS]):
            rts[i % RS].step(band, obands[i % RS], stream=rstreams[i % RS])
    torch.cuda.synchronize()
    barrier()
    for i in range(2 * RS + 3):
        rstep(i)
    barrier()
    ms = timed_batches(rstep, rstreams, Kr)
    ms_med = statistics.median(ms) / Kr
    status = rt.ao.band_status() if mode == "native" else {"error": 0}
    # the full frame on every rank (sum of the zero-padded bands), for the one-GPU time and for the oracle
    full = torch.zeros((RH, RW), dtype=torch.float32, device=dev)
    full[rt.row0:rt.row1] = band
    dist.all_reduce(full)
    ms1 = ms1_serial = None
    ref_dev = torch.empty((RH, RW), dtype=torch.uint8, device=dev)
    if rank == 0:
        ms1, ms1_serial, alg, got = one_gpu(full)           # the N = 1 point, measured in THIS run on rank 0 while the others wait
        if not args.no_cpu:
            from oracle.oracle import Oracle
            ref = Oracle(RW, RH, threads=os.cpu_count() or 1, intensity=INTENSITY).run(full.cpu().numpy())
            ref_dev.copy_(torch.from_numpy(ref))
        else:
            ref_dev.copy_(got)                              # no CPU leg: compare with the one-GPU frame instead
    barrier()
    dist.broadcast(ref_dev, 0)
    rt.step(band, obands[0])
    torch.cuda.synchronize()
    same = torch.tensor([1.0 if torch.equal(ref_dev[rt.row0:rt.row1], obands[0]) else 0.0], dtype=torch.float64, device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    t1 = torch.tensor([ms1 or 0.0, ms1_serial or 0.0, float(alg or 0)], dtype=torch.float64, device=dev)
    dist.broadcast(t1, 0)
    ms1, ms1_serial, alg = float(t1[0]), float(t1[1]), float(t1[2])
    halo = int(rt.ao.halo_bytes(0) + rt.ao.halo_bytes(1))
    del rts, full, ref_dev
    torch.cuda.empty_cache()
    return {"workload": f"{RW}x{RH} single frame, {world} row bands (one per GPU), per-level LowDepth halo rows pushed by peer stores over NVLink inside the step's graph",
            "exchange": mode, "value": round(px / (ms_med * 1e-3) / 1e6, 1), "unit": "Mpixels/s", "steps": Kr, "batches": BATCHES,
            "streams": RS, "ms_per_step": round(ms_med, 5), "batches_ms_per_step": [round(m / Kr, 5) for m in ms], "scaling": "strong", "n_gpus": world,
            "one_gpu_ms_per_frame": round(ms1, 5), "one_gpu_serial_ms_per_frame": round(ms1_serial, 5),
            "speedup_vs_1gpu": round(ms1 / ms_med, 3), "roofline_frac_per_gpu": round(alg / world / (ms_med * 1e-3) / 1e9 / peak, 4),
            "halo_bytes_sent_per_step_rank0": halo, "exchange_error": int(status.get("error", 0)),
            "bands_match_oracle" if not args.no_cpu else "bands_match_single_gpu_frame": bool(same.item() == 1.0)}


def bench_batch1080p(torch, dev, rank, world, throughput, peak, K) -> dict:
    """BASELINE.json configs[4] / SURVEY.md 8d item 3: 64 DISTINCT 1080p frames (camera z-offset 0.25 * frame index), 64 / N per
    GPU, no communication.  A timed batch = `passes` passes over the rank's frames."""
    W, H = WORKLOADS["1080p"]
    total = 64
    per = total // world if total % world == 0 else (total + world - 1) // world
    mine = [f for f in range(rank * per, min(total, (rank + 1) * per))]
    depths = [torch.from_numpy(make_depth(W, H, f)).to(dev) for f in mine]
    outs = [torch.empty((H, W), dtype=torch.uint8, device=dev) for _ in range(len(mine))]
    passes = max(1, (max(K, 64) + len(mine) - 1) // len(mine))
    k = passes * len(mine)
    ms_med, ms, ctxs, _, _ = throughput(W, H, depths, outs, k)
    alg = ctxs[0].algorithmic_bytes(0)
    chk = int(sum(int(o.sum(dtype=torch.int64).item()) for o in outs[:2]))
    agg = W * H * k * world / (ms_med * 1e-3) / 1e6
    return {"workload": f"batch of {total} distinct {W}x{H} frames, {len(mine)} per GPU, throughput mode, no communication",
            "value": round(agg, 1), "unit": "Mpixels/s", "n_gpus": world, "frames_per_gpu": len(mine), "steps_per_gpu": k, "batches": BATCHES,
            "us_per_frame_per_gpu": round(ms_med / k * 1e3, 3), "roofline_frac_per_gpu": round(alg * k / (ms_med * 1e-3) / 1e9 / peak, 4),
            "ao_checksum_rank0_first2": chk, "scaling": "weak"}


def bench_1080p(torch, dev, throughput, serial_ms, peak, K) -> dict:
    W, H = WORKLOADS["1080p"]
    NB = 16                                                     # 16 x 8.3 MB = 133 MB > L2
    depths = [torch.from_numpy(make_depth(W, H, 100 + f)).to(dev) for f in range(NB)]
    outs = [torch.empty((H, W), dtype=torch.uint8, device=dev) for _ in range(NB)]
    k = max(K, 100)
    ms_med, ms, ctxs, _, _ = throughput(W, H, depths, outs, k)
    lat = serial_ms(ctxs[0], depths, outs, k)
    alg = ctxs[0].algorithmic_bytes(0)
    return {"workload": workload_label(W, H), "value": round(W * H * k / (ms_med * 1e-3) / 1e6, 1), "unit": "Mpixels/s",
            "us_per_frame": round(ms_med / k * 1e3, 3), "serial_us_per_frame": round(lat * 1e3, 3),
            "roofline_frac": round(alg * k / (ms_med * 1e-3) / 1e9 / peak, 4), "steps": k, "batches": BATCHES}


def bench_256_single_scale(torch, dev, local, args) -> dict:
    """BASELINE.json configs[0]: 256x256 flat + sphere, SINGLE-SCALE plan (MeaoVariants.single_scale: Downsample -> Render level 1 ->
    final-style Upsample).  The config is the reference's CPU-runnable plumbing case: the scalar CPU twin is timed beside the GPU."""
    from miniengineao_b200 import AmbientOcclusion, Camera, synth
    W = H = 256
    depth = synth.lin01_to_raw(synth.flat_sphere(W, H))
    ao = AmbientOcclusion(Camera(W, H), device=local)
    ao.intensity, ao.singleScale = INTENSITY, True
    d = torch.from_numpy(depth).to(dev)
    o = torch.empty((H, W), dtype=torch.uint8, device=dev)
    for _ in range(5):
        ao.render(d, o)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(200):
        ao.render(d, o)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / 200 * 1e3
    res = {"workload": "256x256 synthetic flat+sphere depth, single-scale AO (Downsample -> Render level 1 -> final-style Upsample)",
           "gpu_us_per_frame": round(us, 3), "gpu_mpix_s": round(W * H / us, 1), "kernels_per_frame": ao.kernels_per_frame}
    if not args.no_cpu:
        from oracle.oracle import Oracle
        orc = Oracle(W, H, threads=1, intensity=INTENSITY, single_scale=True)
        ref = orc.run(depth)
        ts = []
        for _ in range(5):
            t = time.perf_counter(); orc.run(depth); ts.append(time.perf_counter() - t)
        res.update({"cpu_scalar_1thread_ms_per_frame": round(statistics.median(ts) * 1e3, 3),
                    "cpu_scalar_1thread_mpix_s": round(W * H / statistics.median(ts) / 1e6, 2),
                    "gpu_matches_oracle": bool(np.array_equal(ref, o.cpu().numpy())),
                    "note": "the C# twin (host/AmbientOcclusionScalar.cs) cannot be compiled in this image; its line-for-line C twin is what is timed"})
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="4k", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip every CPU-oracle leg (cpu_baseline, oracle checks)")
    ap.add_argument("--quick", action="store_true", help="headline + e2e + roofline only (skip the other configs and the composite)")
    ap.add_argument("--streams", type=int, default=5, help="contexts/streams that frames alternate over in throughput mode")
    ap.add_argument("--band-streams", type=int, default=12, help="band contexts per rank in the row-tiled 8K measurement")
    ap.add_argument("--only-8k", action="store_true", help="development aid: only the 8K single-frame / row-band measurement")
    ap.add_argument("--band-mode", default="native", choices=["native", "p2p"], help="halo exchange: peer stores inside the graph / NCCL send-recv between two graphs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the AO of the last timed step as DIR/ao.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.only_8k:
        ap.error("--dump-outputs covers the headline workload, which --only-8k skips")
    if args.impl == "reference":
        run_reference(args)
    else:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if args.gpus > 1 and world == 1:
            # convenience: relaunch under torchrun
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
            raise SystemExit(subprocess.call(cmd))
        run_ours(args)


if __name__ == "__main__":
    main()
