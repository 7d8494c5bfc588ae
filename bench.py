#!/usr/bin/env python
"""bench.py -- encode+decode throughput of the HGI hot path on B200 (BASELINE.json metric).

Workload (BASELINE.json configs[4], the largest single-GPU configuration; weak scaling): per GPU
a batch of 4096 synthetic 1920x1080 8-bit frames, frame k = (x*y + 31k) & 255 (frame 0 is the
reference's criterion bench image, benches/bench.rs:24-28), level = 4, interpolator Crossed,
quantizator Linear at Lossless and at Medium.  One *step* = for q in (Lossless, Medium):
Encoder::encode over the batch, then Decoder::decode over the batch.  `value` counts every pixel
once per encode+decode round trip: Mpixel/s = n_gpus * 2 * frames * 1920*1080 / step_time.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Timed with CUDA events on the launching stream after W warm-up steps, barrier + synchronize on
both sides, max over ranks.  The working set (8.5 GB per plane set) is far larger than the 126 MB
L2, so no flush is needed between iterations.  `e2e` is the same metric through the host-pointer
C-ABI calls (pinned host buffers, H2D + D2H inside the timed region).  `--impl reference` times
the CPU restatement of the reference (oracle/, all host threads) on a bounded sample.

`--dump-outputs DIR` writes what the last timed step returned (rank 0's grids and decoded planes at both quantizers)
as float32 .npy files: a fixed, seeded sample, so two builds run with the same arguments compare output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, LEVELS = 1920, 1080, 4
QLEVELS = (0, 2)                      # Lossless, Medium
FRAMES_PER_GPU = 4096
METRIC = "encode+decode Mpixel/s"
UNIT = "Mpixel/s"


def workload_config(frames, n_gpus):
    return {"workload": f"batch of {frames} synthetic 1080p frames per GPU, Lossless+Medium, level=4, Crossed "
                        f"(BASELINE configs[4]; image-sharded, {n_gpus} GPU(s))",
            "frames_per_gpu": frames, "width": W, "height": H, "levels": LEVELS,
            "quantizators": ["Lossless", "Medium"], "interpolator": "Crossed", "parallelism": f"image-shard x{n_gpus}",
            "l2_policy": "inputs (8.5 GB per plane set) >> 126 MB L2; no flush needed"}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profiled_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: in-process NVML every 5 ms (a thread; the main
    thread sits in cudaDeviceSynchronize with the GIL released), `nvidia-smi -lms` as the fallback -- its piped output
    arrives in bursts, which loses short timed regions."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
            0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nvml, self.stop_flag = index, [], None, None, False

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            pr = torch.cuda.get_device_properties(self.index)
            bus = f"{pr.pci_domain_id:08X}:{pr.pci_bus_id:02X}:{pr.pci_device_id:02X}.0"
            return pynvml, pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)

    def start(self):
        try:
            self.nvml = self._nvml_handle()
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv, h = self.nvml
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = 0
        while not self.stop_flag:
            try:
                clk = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                flags = ["Active" if mask & bit else "Not Active" for bit in (0x8, 0x40, 0x20, 0x4)]
                self.rows.append((time.time(), [str(self.index), str(clk), str(mx), "", hex(mask)] + flags))
            except Exception:
                pass
            time.sleep(0.005)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=0.0, t1=float("inf")):
        """Summary of the samples that arrived in the host-time window [t0, t1]."""
        self.stop_flag = True
        if self.nvml is None and not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"]}
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(5)
            except Exception:
                self.proc.kill()
        slack = 0.06 if self.proc else 0.0
        sm, mx, reasons = [], [], set()
        for ts, r in self.rows:
            if not (t0 <= ts <= t1 + slack):
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "source": "nvml" if self.nvml else "nvidia-smi", "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path (its C restatement, oracle/ -- the
    reference is nightly Rust and cannot be built here), all host threads, bounded sample."""
    if rank != 0:
        return
    import numpy as np
    from oracle import c as oc
    threads = oc.max_threads()
    sample = max(threads * 2, 32)
    yy, xx = np.mgrid[0:H, 0:W]
    frames = np.stack([((xx * yy + 31 * k) & 255).astype(np.uint8) for k in range(sample)])

    def step():
        for q in QLEVELS:
            grids = oc.encode_batch(frames, LEVELS, qlevel=q, n_threads=threads)
            oc.decode_batch(grids, LEVELS, n_threads=threads)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    value = len(QLEVELS) * sample * W * H / dt / 1e6
    desc = f"{sample} of the workload's 1080p frames per step, by-image pthreads"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(FRAMES_PER_GPU, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def cpu_baseline(budget_s=12.0):
    import numpy as np
    from oracle import c as oc
    threads = oc.max_threads()
    sample = max(threads * 2, 32)
    yy, xx = np.mgrid[0:H, 0:W]
    frames = np.stack([((xx * yy + 31 * k) & 255).astype(np.uint8) for k in range(sample)])
    reps, t0 = 0, time.perf_counter()
    while True:
        for q in QLEVELS:
            grids = oc.encode_batch(frames, LEVELS, qlevel=q, n_threads=threads)
            oc.decode_batch(grids, LEVELS, n_threads=threads)
        reps += 1
        if time.perf_counter() - t0 > budget_s or reps >= 50:
            break
    dt = (time.perf_counter() - t0) / reps
    # single-thread figure = the reference's own execution model (one image, one thread)
    t1 = time.perf_counter()
    g = oc.encode(frames[0], LEVELS, qlevel=2)
    oc.decode(g, LEVELS)
    st = time.perf_counter() - t1
    return {"value": len(QLEVELS) * sample * W * H / dt / 1e6, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{sample} of the workload's 1080p frames x {reps} reps, by-image pthreads, oracle/hgi_oracle.c",
            "single_thread_value": W * H / st / 1e6}


def bind_to_gpu_numa_node(local_rank):
    """Run this rank (and first-touch its pinned buffers) on the NUMA node its GPU hangs off, so that 8 ranks
    streaming over PCIe do not all pull through one socket.  Best effort; returns a note for the JSON line."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id       # e.g. 0000:1B:00.0
        if isinstance(bus, int):
            return None
        base = f"/sys/bus/pci/devices/{bus.lower()}"
        node = int(open(base + "/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception:
        return None


def oracle_parity(frames, encs, dec, ctx, n_check=64):
    """After the timed steps, outside the timed region: `n_check` frames spread over rank 0's shard are encoded and
    decoded again at both quantizers and compared BYTE FOR BYTE with the oracle (grid and decoded plane)."""
    import numpy as np
    import torch
    from oracle import c as oc
    n = frames.shape[0]
    idx = sorted(set(int(round(i * (n - 1) / max(1, n_check - 1))) for i in range(min(n_check, n))))
    sel = torch.tensor(idx, device=frames.device)
    sub = frames.index_select(0, sel).contiguous()
    host = sub.cpu().numpy()
    bad, compared = 0, 0
    for enc, q in zip(encs, QLEVELS):
        g = enc.encode_device(sub)
        r = dec.decode_device(LEVELS, g)
        torch.cuda.synchronize()
        want_g = oc.encode_batch(host, LEVELS, qlevel=q, n_threads=oc.max_threads())
        want_r = oc.decode_batch(want_g, LEVELS, n_threads=oc.max_threads())
        bad += int((g.cpu().numpy() != want_g).sum()) + int((r.cpu().numpy() != want_r).sum())
        compared += 2 * host.size
    return {"frames_checked": len(idx), "quantizators": ["Lossless", "Medium"], "bytes_compared": compared,
            "mismatches": bad, "checker": "oracle/hgi_oracle.c (grid bytes and decoded planes, every byte)"}


DUMP_SEED, DUMP_PIXELS = 20261020, 1 << 20


def dump_positions(n):
    """What --dump-outputs keeps of a batch of n frames: one frame index, and DUMP_PIXELS flat (frame, y, x) indices
    over the whole batch.  Seeded, so the same arguments give the same positions in every run and every build."""
    import numpy as np
    rng = np.random.default_rng(DUMP_SEED)
    return int(rng.integers(n)), np.sort(rng.integers(0, n * H * W, DUMP_PIXELS))


def dump_outputs(out_dir, outputs):
    """`outputs`: name -> (n, H, W) uint8 CUDA tensor.  Writes <name>_frame.npy (the chosen frame in full) and
    <name>_sample.npy (the sampled pixels) as float32: 12.5 MB per output at 1080p, 50 MB for the four."""
    import numpy as np
    import torch
    first = next(iter(outputs.values()))
    frame, pix = dump_positions(first.shape[0])
    pix = torch.from_numpy(pix).to(first.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, f"{name}_frame.npy"), t[frame].cpu().numpy().astype(np.float32))
        np.save(os.path.join(out_dir, f"{name}_sample.npy"), t.reshape(-1)[pix].cpu().numpy().astype(np.float32))


def time_events(fn, stream, reps, warm=3):
    import torch
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(reps):
        fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b) / reps        # ms


def per_call_us(fn, calls=200, reps=5):
    """GPU-side cadence of `calls` back-to-back device-API calls replayed from one torch CUDA graph (no interpreter
    between the launches): us per call."""
    import torch
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            fn(s)
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            for _ in range(calls):
                fn(s)
        best = None
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(s)
            g.replay()
            b.record(s)
            b.synchronize()
            t = a.elapsed_time(b) * 1e3 / calls
            best = t if best is None else min(best, t)
    torch.cuda.current_stream().wait_stream(s)
    return best


def extra_block(hgi, ctx, dev, rank, world, dist, peak, grids_medium, barrier):
    """Numbers the headline line does not carry: single planes (configs[1..3] per call), configs[3] (16384^2, level 8,
    Medium) on one GPU and as row bands over the ranks, and the residual histogram -- all device-resident."""
    import torch
    Qm = hgi.QuantizationLevel
    out = {}
    stream = torch.cuda.current_stream(dev)
    # ---- residual histogram over this rank's Medium grids: 1 B/byte read
    n = grids_medium.shape[0]
    hist = torch.empty((n, 256), dtype=torch.int32, device=dev)
    L = hgi.lib()
    sth = stream.cuda_stream or 1
    ms = time_events(lambda: ctx.check(L.hgi_histogram_dev(ctx._h, grids_medium.data_ptr(), H * W, n, hist.data_ptr(), sth), "hist"), stream, 10)
    assert int(hist[0].sum().item()) == H * W
    gbs = n * H * W / (ms * 1e-3) / 1e9
    out["histogram"] = {"kernel": "hgi_hist_kernel (256-bin per image, private per-lane columns in shared memory)",
                        "frames": n, "ms": ms, "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s",
                                                           "frac": gbs / peak, "algorithmic_bytes_per_byte": 1.0}}
    if rank == 0:
        # ---- single planes, us per device-resident call (configs[1]: 1920x1080 L4; configs[2] size: 2368x2614 L6 High)
        single = {}
        for name, (w, h, lv, q) in {"c2_1080p_L4_lossless": (1920, 1080, 4, 0), "c2_1080p_L4_medium": (1920, 1080, 4, 2),
                                    "c3_2368x2614_L6_high": (2368, 2614, 6, 3)}.items():
            yy = torch.arange(h, device=dev, dtype=torch.int32)[:, None]
            xx = torch.arange(w, device=dev, dtype=torch.int32)[None, :]
            img = ((xx * yy) & 255).to(torch.uint8).contiguous()
            g, o = torch.empty_like(img), torch.empty_like(img)
            enc = hgi.Encoder(hgi.Crossed, hgi.Linear(Qm(q)), lv, ctx=ctx)
            dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
            single[name] = {"encode_us_per_call": per_call_us(lambda s: enc.encode_device(img, grids_out=g, stream=s.cuda_stream)),
                            "decode_us_per_call": per_call_us(lambda s: dec.decode_device(lv, g, images_out=o, stream=s.cuda_stream))}
        out["single_plane"] = dict(single, method="200 back-to-back hgi_*_dev calls replayed from one CUDA graph, best of 5")
    # ---- configs[3]: 16384 x 16384, level 8, Medium
    n16, lv = 16384, 8
    enc = hgi.Encoder(hgi.Crossed, hgi.Linear(Qm.Medium), lv, ctx=ctx)
    dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
    xx = torch.arange(n16, device=dev, dtype=torch.int32)[None, :]
    st = torch.cuda.Stream(dev)                       # a real stream: the launch chain is replayed from a graph
    if rank == 0:
        yy = torch.arange(n16, device=dev, dtype=torch.int32)[:, None]
        img = ((xx * yy) & 255).to(torch.uint8).contiguous()
        g, o = torch.empty_like(img), torch.empty_like(img)
        torch.cuda.synchronize()
        with torch.cuda.stream(st):
            te = time_events(lambda: enc.encode_device(img, grids_out=g, stream=st.cuda_stream), st, 20) * 1e3
            td = time_events(lambda: dec.decode_device(lv, g, images_out=o, stream=st.cuda_stream), st, 20) * 1e3
        err = int((o[::64].to(torch.int16) - img[::64].to(torch.int16)).abs().max().item())
        assert err <= 20 and torch.equal(o[::256, ::256], img[::256, ::256])
        px = float(n16) * n16
        out["c4_16384_L8_medium_1gpu"] = {"encode_us": te, "decode_us": td,
                                          "encode_frac_of_peak": 2 * px / (te * 1e-6) / 1e9 / peak,
                                          "decode_frac_of_peak": 2 * px / (td * 1e-6) / 1e9 / peak,
                                          "graph_launches": ctx.graph_launches}
        del img, g, o
    if world > 1:
        # row bands: rank r owns band r (heights multiples of 256, 257 overlap rows), no exchange
        bands = hgi.sharding.plan_bands(n16, lv, world)
        t_ms = -1.0
        if rank < len(bands):
            bd = bands[rank]
            yy = torch.arange(bd.y0, bd.in_y1, device=dev, dtype=torch.int32)[:, None]
            bimg = ((xx * yy) & 255).to(torch.uint8).contiguous()
            bg, bo = torch.empty_like(bimg), torch.empty_like(bimg)

            def band_step():
                enc.encode_device(bimg, grids_out=bg, stream=st.cuda_stream)
                dec.decode_device(lv, bg, images_out=bo, stream=st.cuda_stream)
            torch.cuda.synchronize()
            barrier()
            with torch.cuda.stream(st):
                t_ms = time_events(band_step, st, 50, warm=5)
        else:
            barrier()
        t = torch.tensor([t_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if rank == 0:
            one = out["c4_16384_L8_medium_1gpu"]
            out["c4_row_bands"] = {"ranks": world, "bands": len(bands), "encode_plus_decode_us": float(t.item()) * 1e3,
                                   "vs_1gpu": (one["encode_us"] + one["decode_us"]) / (float(t.item()) * 1e3),
                                   "rows_in_per_rank": bands[0].rows_in, "rows_out_per_rank": bands[0].rows_out,
                                   "timing": "max over ranks, CUDA events over 50 encode+decode pairs per rank"}
    return out


def run_ours(args, rank, world, local_rank):
    import torch
    import rustyhgi_b200 as hgi

    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        # NCCL_DEBUG is whatever the launcher set; only its log file defaults to stderr so that stdout stays the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    frames_n = args.frames
    ctx = hgi.Context(local_rank, int(os.environ.get("HGI_BENCH_PATH", "0")))   # 0 = default path (tuning hook)
    encs = [hgi.Encoder(hgi.Crossed, hgi.Linear(hgi.QuantizationLevel(q)), LEVELS, ctx=ctx) for q in QLEVELS]
    dec = hgi.Decoder(hgi.Crossed, ctx=ctx)

    yy = torch.arange(H, device=dev, dtype=torch.int32)[:, None]
    xx = torch.arange(W, device=dev, dtype=torch.int32)[None, :]
    frames = torch.empty((frames_n, H, W), dtype=torch.uint8, device=dev)
    first = rank * frames_n                                 # global frame index of this rank's shard
    for k0 in range(0, frames_n, 256):
        k = torch.arange(first + k0, first + min(k0 + 256, frames_n), device=dev, dtype=torch.int32)[:, None, None]
        frames[k0:k0 + k.shape[0]] = ((xx * yy + 31 * k) & 255).to(torch.uint8)
    # one grid and one decoded batch per quantizer, so that the last step leaves every output it computed intact
    grids = [torch.empty_like(frames) for _ in QLEVELS]
    backs = [torch.empty_like(frames) for _ in QLEVELS]
    stream = torch.cuda.current_stream(dev)

    ev = lambda: torch.cuda.Event(enable_timing=True)
    marks = []

    def step(record):
        row = [ev() for _ in range(2 * len(QLEVELS) + 1)] if record else None
        if record:
            row[0].record(stream)
        for i, enc in enumerate(encs):
            enc.encode_device(frames, grids_out=grids[i])
            if record:
                row[2 * i + 1].record(stream)
            dec.decode_device(LEVELS, grids[i], images_out=backs[i])
            if record:
                row[2 * i + 2].record(stream)
        if record:
            marks.append(row)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                                     # started early: nvidia-smi takes a while to come up
    for _ in range(args.warmup):
        step(False)
    barrier()
    wall0 = time.time()
    launches0 = ctx.kernel_launches
    t_begin, t_end = ev(), ev()
    t_begin.record(stream)
    for _ in range(args.steps):
        step(True)
    t_end.record(stream)
    barrier()
    clocks = sampler.stop(wall0, time.time()) if rank == 0 else None
    launches = ctx.kernel_launches - launches0
    elapsed_ms = t_begin.elapsed_time(t_end)
    if dist:
        t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    px_step = len(QLEVELS) * frames_n * W * H
    value = world * px_step / (ms_per_step * 1e-3) / 1e6

    # per-kernel durations (L=4 => each encode / decode is exactly one kernel launch)
    names = ["encode_lossless", "decode_lossless", "encode_medium", "decode_medium"]
    per = {n: statistics.mean(r[i].elapsed_time(r[i + 1]) for r in marks) for i, n in enumerate(names)}

    # sanity: the timed outputs are real (Medium): bounded error, seeds raw
    err = int((backs[1][:8].to(torch.int16) - frames[:8].to(torch.int16)).abs().max().item())
    assert err <= 20 and torch.equal(backs[1][:8, ::16, ::16], frames[:8, ::16, ::16]), "bench output failed sanity"

    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {f"{kind}_{qname}": t for qname, g, b in zip(("lossless", "medium"), grids, backs)
                                         for kind, t in (("grid", g), ("decoded", b))})

    # ---- strong scaling of the workload as BASELINE configs[4] words it: 4096 frames in total, 4096 / N per rank ----
    strong = None
    if world > 1 and not args.no_extra:
        share = max(1, frames_n // world)
        fs, gs, bs = frames[:share], grids[1][:share], backs[1][:share]

        def strong_step():
            for enc in encs:
                enc.encode_device(fs, grids_out=gs)
                dec.decode_device(LEVELS, gs, images_out=bs)
        barrier()
        ms = time_events(strong_step, stream, args.steps)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        strong = {"frames_total": share * world, "frames_per_gpu": share, "ms_per_step": float(t.item()),
                  "value": len(QLEVELS) * share * world * W * H / (float(t.item()) * 1e-3) / 1e6, "unit": UNIT,
                  "note": "the same step over 4096 / N frames per rank (BASELINE configs[4] as written); max over ranks"}

    # ---- full parity of sampled frames against the oracle (rank 0; outside every timed region) ----
    parity = None
    if rank == 0 and not args.no_cpu:
        parity = oracle_parity(frames, encs, dec, ctx)
        assert parity["mismatches"] == 0, f"bench outputs differ from the oracle: {parity}"

    extra = None
    if not args.no_extra:
        try:
            extra = extra_block(hgi, ctx, dev, rank, world, dist, measured_peak()[0], grids[1], barrier)
        except Exception as exc:                                   # the headline line must survive a failing side measurement
            if world > 1:
                raise                                              # ranks would lose step with each other: fail loudly instead
            extra = {"error": f"{type(exc).__name__}: {exc}"}
        if strong:
            extra["strong_scaling"] = strong

    # ---- e2e: host-pointer C-ABI calls, pinned host memory, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        del backs
        torch.cuda.empty_cache()
        n_e = min(args.e2e_frames or 1024, frames_n)        # pinned buffer size (frames); see e2e_step
        n_sub = -(-frames_n // n_e)                         # sub-batches per step: the whole workload streams through
        try:
            h_in = torch.empty((n_e, H, W), dtype=torch.uint8, pin_memory=True)
            h_grid = torch.empty((n_e, H, W), dtype=torch.uint8, pin_memory=True)
            h_out = torch.empty((n_e, H, W), dtype=torch.uint8, pin_memory=True)
        except Exception as exc:                            # pinned allocation refused: say so
            h_in = None
            e2e = {"value": None, "unit": UNIT, "error": f"pinned allocation failed: {exc}"}
        if h_in is not None:
            h_in.copy_(frames[:n_e])
            torch.cuda.synchronize()
            a_in, a_grid, a_out = h_in.numpy(), h_grid.numpy(), h_out.numpy()
            import ctypes
            L = hgi.lib()

            def e2e_step():
                # the step's frames_n frames go through the host API as n_sub calls on one pinned
                # buffer set of n_e frames (host RAM on the box is 196 GB for 8 ranks)
                for enc in encs:
                    p = enc._p()
                    for _ in range(n_sub):
                        ctx.check(L.hgi_encode_batch_u8(ctx._h, a_in.ctypes.data, n_e, W, H, ctypes.byref(p),
                                                        a_grid.ctypes.data, None), "hgi_encode_batch_u8")
                        ctx.check(L.hgi_decode_batch_u8(ctx._h, a_grid.ctypes.data, n_e, W, H, ctypes.byref(p),
                                                        a_out.ctypes.data), "hgi_decode_batch_u8")

            e_steps = max(1, min(args.steps, 3))
            e2e_step()                                      # warm-up (allocates the staging slots)
            barrier()
            t0 = time.perf_counter()
            for _ in range(e_steps):
                e2e_step()
            barrier()
            dt = (time.perf_counter() - t0) / e_steps
            if dist:
                t = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            assert int((h_out[:4].to(torch.int16) - h_in[:4].to(torch.int16)).abs().max().item()) <= 20
            f_e = n_sub * n_e
            bytes_dir = len(QLEVELS) * 2 * f_e * W * H      # encode in + decode in / encode out + decode out
            e2e = {"value": world * len(QLEVELS) * f_e * W * H / dt / 1e6, "unit": UNIT,
                   "h2d_bytes_per_step": bytes_dir, "d2h_bytes_per_step": bytes_dir, "frames_per_gpu": f_e,
                   "pinned_buffer_frames": n_e,
                   "steps": e_steps, "ms_per_step": dt * 1e3, "numa_binding": numa,
                   "api": "hgi_encode_batch_u8 + hgi_decode_batch_u8 (host pointers, pinned)"}

    if rank == 0:
        peak, peak_src = measured_peak()
        alg_bytes = 2.0 * frames_n * W * H                  # 2 B/pixel: read pixel + write residual
        dom = "encode_medium"
        achieved = alg_bytes / (per[dom] * 1e-3) / 1e9
        traffic = profiled_traffic()
        roofline = {"bound": "hbm", "kernel": "hgi_tile_fast_part_kernel<encode, Crossed, Linear> (Medium): interior-tile launch + right-tile-column "
                              "launch + bottom-tile-row launch of one encode, timed together",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "peak_source": peak_src, "frac_of_nominal_8TBs": achieved / 8000.0,
                    "algorithmic_bytes_per_launch": alg_bytes,
                    "ms_per_launch": per[dom],
                    "traffic": traffic["dram_bytes_per_pixel"] * frames_n * W * H if traffic else None,
                    "traffic_source": traffic.get("source") if traffic else None,
                    "per_kernel": {n: {"ms": per[n], "GB/s": alg_bytes / (per[n] * 1e-3) / 1e9,
                                       "frac": alg_bytes / (per[n] * 1e-3) / 1e9 / peak} for n in names},
                    "step": {"algorithmic_bytes": alg_bytes * len(names), "GB/s": alg_bytes * len(names) / (ms_per_step * 1e-3) / 1e9,
                             "frac": alg_bytes * len(names) / (ms_per_step * 1e-3) / 1e9 / peak}}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(frames_n, world),
                "roofline": roofline, "cpu_baseline": None if args.no_cpu else cpu_baseline(), "e2e": e2e,
                "gpu_launches": int(launches), "clocks": clocks, "parity": parity, "extra": extra}
        print(json.dumps(line), flush=True)
    ctx.close()
    if dist:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=FRAMES_PER_GPU, help="frames per GPU (default: the named workload)")
    ap.add_argument("--e2e-frames", type=int, default=0, help="frames in the pinned e2e buffers (default 1024)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra block (single planes, config 4, histogram, strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's outputs to DIR "
                                                          "as float32 .npy files (50 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1 and "RANK" not in os.environ:
        # launched without torchrun: start one rank per GPU ourselves
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
