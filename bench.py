#!/usr/bin/env python3
"""bench.py -- interpolated frames/sec of the RIFE hot path (BASELINE.json metric) on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload 1080p|4k] [--impl ours|reference] [--scaling weak|strong]
                  [--dump-outputs DIR]

A step = one pass of the hot path over one batch of synthetic frame pairs (rife-v4.6, t = 0.5): 128 pairs of 1080p, 32 of 4K.
One invocation measures BOTH resolutions of the metric: the headline keys are BASELINE configs[1] (1920x1080), and
`also["4k"]` carries the same measurements for configs[2] (3840x2160) -- unless --workload 4k makes 4K the headline.
  value     whole-job frames/s with the frames resident in HBM (rife_b200_process_batch_device), CUDA-event timed on the
            stream the kernels are launched on, max over ranks.
  e2e       the same metric through the batch call with HOST buffers (rife_b200_process_batch, pinned memory): H2D of the
            frames + D2H of the results inside the timed region.
  e2e_process  frames/s through rife_b200_process -- the ONLY call the reference's caller makes (src/main.cpp:360) -- from
            1, 2 (the reference default -j 1:2:2) and 8 caller threads on one handle, pageable and pinned buffers (N = 1 only).
  parity    the oracle's frame for one pair of the workload against what the timed configuration (lock-step batch, lanes)
            produces for it: PSNR, max |diff| in LSB, share of differing values.  The run FAILS (exit code 3) if max > 1 LSB or
            PSNR <= 50 dB (BASELINE.json north_star).
  roofline  the dominant kernel (tcgen05 conv3x3 64->64 at quarter resolution, 44 % of the model's FLOPs): `achieved` is
            measured IN the step -- CUDA events around the eight back-to-back launches of IFBlock 3's residual chain, on
            the lane's stream (option "ktime") -- and, beside it, the same kernel timed alone; 2*9*Cin*Cout*H*W FLOP per
            launch / time; peak = measured cuBLAS bf16 TF/s.  `stages` is the per-stage breakdown of one lock-step batch.
  cpu_baseline  the reference's own CPU path (oracle/_ref: its rife.cpp CPU functions + vendored ncnn) on the host cores,
            bounded sample, rank 0 only.
--dump-outputs DIR writes, per measured resolution, what the timed path returned in its last step: DIR/<workload>_frames_sample.npy,
            float32, the values of a fixed sample (seed 0, DUMP_SAMPLE positions drawn with replacement, in ascending order) of
            the step's interpolated frames, all pairs of rank 0 stacked as [pair, y, x, rgb] and flattened.  The frames are seeded
            (synth.stream), so two builds run with the same arguments can be compared value for value.
--impl reference times that CPU path alone on the same workload (the driver computes the ratio).
Multi-GPU: one process per GPU (torchrun); frame pairs are independent, so ranks share nothing after rank 0 broadcasts the
packed model over NCCL.  --scaling weak (default): fixed pairs per GPU.  --scaling strong: ONE fixed stream (256 pairs of
4K / 1024 of 1080p) cut into contiguous shards by dist_util.shard_pairs (BASELINE configs[2]: "batch sharded across 8xB200").
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {"1080p": (1920, 1080, "rife-v4.6 1920x1080 synthetic frame-pair stream (BASELINE configs[1])"),
             "4k": (3840, 2160, "rife-v4.6 3840x2160 UHD-flag stream (BASELINE configs[2]; -u is a no-op for v4 nets)")}
GFLOP_PER_FRAME = {"1080p": 175.2, "4k": 701.0}  # BASELINE.md section 2
PAIRS_DEFAULT = {"1080p": 128, "4k": 32}
STRONG_STREAM = {"1080p": 1024, "4k": 256}       # --scaling strong: pairs of the one fixed stream
PAIRS_ENV = int(os.environ.get("RIFE_BENCH_PAIRS", "0"))  # profiling runs shrink the step
DISTINCT_FRAMES = 129  # consecutive frames of the synthetic stream: the default steps (128 / 32 pairs) never send a frame twice as
# a NEW frame -- pair i is (frame i, frame i + 1), so the host-buffer leg uploads pairs + 1 distinct frames per step, what a real
# stream needs (with 9 cycling frames, as until round 2, the library's per-call frame table reduced the upload to 9 frames)
MODEL = "rife-v4.6"
DUMP_SAMPLE = 4 << 20  # values per resolution written by --dump-outputs: 16 MiB of float32 each, 32 MiB for both


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"


def _physical_index(idx):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        parts = [p for p in vis.split(",") if p.strip()]
        if idx < len(parts) and parts[idx].strip().isdigit():
            return int(parts[idx])
    return idx


def bind_to_gpu_numa(local):
    """Pin this process (and so its pinned host buffers, first touch) to the CPUs next to its GPU.  Best effort; returns a note."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(_physical_index(local))
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(":", 1)
        path = "/sys/bus/pci/devices/%s:%s/local_cpulist" % (dom[-4:].lower(), rest.lower())
        cpus = set()
        for part in open(path).read().strip().split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "no local cpus"
        os.sched_setaffinity(0, cpus)
        node = open(path.replace("local_cpulist", "numa_node")).read().strip()
        return "cpus of numa node %s (%d)" % (node, len(cpus))
    except Exception as e:
        return "not bound (%s)" % str(e)[:60]


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML in-process, every 100 ms;
    falls back to nvidia-smi when pynvml is unavailable)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, idx):
        super().__init__(daemon=True)
        self.idx, self.sm, self.mx, self.reasons, self.stop_flag = idx, [], None, set(), False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(_physical_index(idx))
            self.mx = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nvml = None

    def run(self):
        # 100 ms: polling NVML every 5 ms stalled this process's own cudaMemcpyAsync calls by 10-250 ms now and then (the e2e leg
        # dropped from ~2150 to 1000-1800 frames/s, profiles/r2_s17_sampler_stall.txt); 0 = no sampling (diagnosis only)
        period = float(os.environ.get("RIFE_BENCH_SAMPLER_MS", "100")) / 1000.0
        if period <= 0:
            return
        while not self.stop_flag:
            try:
                if self.nvml:
                    self.sm.append(self.nvml.nvmlDeviceGetClockInfo(self.h, self.nvml.NVML_CLOCK_SM))
                    try:
                        r = self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        r = self.nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    for bit, name in self.REASONS.items():
                        if r & bit:
                            self.reasons.add(name)
                    time.sleep(period)
                else:
                    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
                    o = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                       stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5).stdout.strip()
                    if o:
                        r = [x.strip() for x in o.split(",")]
                        if r[0].isdigit():
                            self.sm.append(int(r[0]))
                        if r[1].isdigit():
                            self.mx = int(r[1])
                        for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[2:6]):
                            if v.lower().startswith("active"):
                                self.reasons.add(name)
                    time.sleep(0.1)
            except Exception:
                time.sleep(0.05)

    def summary(self):
        self.stop_flag = True
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.mx, "reasons": sorted(self.reasons), "samples": len(sm)}


def cpu_reference(workload, frames, threads=None, warmup=1):
    """Times the reference's CPU path on `frames` frames of the workload; returns (dict for the JSON line, the oracle's frame)."""
    import parity
    w, h, _ = WORKLOADS[workload]
    a, b = parity.synth.pair(w, h)
    ncpu = os.cpu_count() or 1
    if threads is None:
        # the reference's OpenMP scaling is not monotonic (measured on the 128-thread B200 host: 16 threads 1.11 s/frame,
        # 32: 1.27, 64: 2.2, 128: 10.5 at 1080p -- profiles/r1_cpu_thread_sweep.txt): pick the best of a short sweep at 1080p
        best = None
        sw, sh, _ = WORKLOADS["1080p"]
        sa, sb = (a, b) if workload == "1080p" else parity.synth.pair(sw, sh)
        for t in sorted({min(ncpu, c) for c in (8, 16, 32)}):
            _, i = parity.run_oracle(MODEL, sa, sb, 0.5, threads=t, repeat=1, warmup=0)
            if best is None or i["sec_per_frame"][0] < best[1]:
                best = (t, i["sec_per_frame"][0])
        threads = best[0]
    frame, info = parity.run_oracle(MODEL, a, b, 0.5, threads=threads, repeat=frames, warmup=warmup)
    secs = info["sec_per_frame"]
    fps = len(secs) / sum(secs)
    return {"value": fps, "unit": "frames/s", "cores": threads, "kind": info["kind"],
            "sample": "%d frames of %s after %d warm-up (%.2f s/frame)" % (len(secs), workload, warmup, sum(secs) / len(secs))}, frame


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    w, h, desc = WORKLOADS[args.workload]
    frames = 2 if args.workload == "1080p" else 1
    t0 = time.time()
    per_step = []
    base = None
    first, _ = cpu_reference(args.workload, 1, warmup=0)  # also picks the thread count
    for _ in range(args.steps):
        base, _ = cpu_reference(args.workload, frames, threads=first["cores"], warmup=0)
        per_step.append(base["value"])
        if time.time() - t0 > 240:
            break
    fps = sum(per_step) / len(per_step)
    base["value"] = fps
    base["sample"] = "each step = %d frames of %s; %d steps" % (frames, args.workload, len(per_step))
    line = {"impl": "reference", "metric": "interpolated frames/sec (rife-v4.6)", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": len(per_step), "warmup": args.warmup, "ms_per_step": 1000.0 * frames / fps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": desc, "timestep": 0.5},
            "cpu_baseline": base, "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


class Ctx:
    pass


def host_link_gbs():
    """Measured rate of this GPU's host link with pinned memory (256 MiB copies, CUDA events, best of 3 per direction): the bound
    of the e2e legs, which move 6.2 MB (1080p) / 24.9 MB (4K) of result per frame device -> host."""
    import torch
    n = 256 << 20
    h = torch.empty(n, dtype=torch.uint8).pin_memory()
    d = torch.empty(n, dtype=torch.uint8, device="cuda")
    out = {}
    for name, (dst, src) in (("h2d", (d, h)), ("d2h", (h, d))):
        best = None
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dst.copy_(src, non_blocking=True)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None or ms < best else best
        out[name] = round(n / (best * 1e-3) / 1e9, 1)
    return out


def dump_outputs(out_dir, workload, out_dev):
    """The fixed sample of the frames in `out_dev` (device tensors, one per pair) described in the module docstring."""
    import numpy as np
    import torch
    flat = torch.stack(out_dev).view(-1)
    idx = np.sort(np.random.default_rng(0).integers(0, flat.numel(), min(DUMP_SAMPLE, flat.numel())))
    vals = flat[torch.from_numpy(idx).to(flat.device)].to(torch.float32).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "%s_frames_sample.npy" % workload), vals)


def measure(ctx, workload, args, headline):
    """All GPU-side measurements of one resolution.  Returns a dict (rank-local; times are already max-reduced over ranks)."""
    import torch
    import parity
    pkg, eng, dist, world, rank, local = ctx.pkg, ctx.eng, ctx.dist, ctx.world, ctx.rank, ctx.local
    w, h, desc = WORKLOADS[workload]
    if args.scaling == "strong":
        sys.path.insert(0, os.path.join(ROOT, "rife-ncnn-vulkan_b200"))
        import dist_util
        total = PAIRS_ENV if PAIRS_ENV > 0 else STRONG_STREAM[workload]
        lo, hi = dist_util.shard_pairs(total, world, rank)
        pairs, first_pair, total_pairs = hi - lo, lo, total
    else:
        pairs = PAIRS_ENV if PAIRS_ENV > 0 else PAIRS_DEFAULT[workload]
        first_pair, total_pairs = 0, pairs * world
    res = {"pairs_per_step_this_rank": pairs, "pairs_per_step_all_ranks": total_pairs}

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # synthetic frames: a short stream (distinct per rank under weak scaling; one shared stream under strong scaling)
    nframes = min(max(pairs, 1), DISTINCT_FRAMES - 1) + 1
    seed = rank if args.scaling == "weak" else 0
    frames = parity.synth.stream(first_pair, nframes, w, h, seed=seed)
    host = [torch.from_numpy(f).pin_memory() for f in frames]
    dev = [t.cuda(non_blocking=True) for t in host]
    out_dev = [torch.empty_like(dev[0]) for _ in range(pairs)]
    out_host = [torch.empty_like(host[0]).pin_memory() for _ in range(pairs)]
    stream = ctx.stream
    eng.set_stream(stream.cuda_stream)
    eng.set_option("async", 1)
    torch.cuda.synchronize()
    d_in0 = [dev[i % (nframes - 1)].data_ptr() for i in range(pairs)]
    d_in1 = [dev[i % (nframes - 1) + 1].data_ptr() for i in range(pairs)]
    d_out = [t.data_ptr() for t in out_dev]
    ts = [args.timestep] * pairs

    def step_device():
        if pairs:
            eng.process_batch_ptr(d_in0, d_in1, w, h, ts, d_out, device=True)

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step_device()
        barrier()
        launches0 = pkg.launch_count()
        sampler = ClockSampler(local)
        sampler.start()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for k in range(args.steps):
            ctx.l2_flush.zero_()  # flush L2 between timed iterations (outside the event bracket)
            ev[k][0].record(stream)
            step_device()
            ev[k][1].record(stream)
        barrier()
        res["gpu_launches"] = int(pkg.launch_count() - launches0)
    if args.dump_outputs and rank == 0 and pairs:
        dump_outputs(args.dump_outputs, workload, out_dev)
    ms_total = reduce_max(sum(a.elapsed_time(b) for a, b in ev))
    res["ms_per_step"] = ms_total / args.steps
    res["value"] = total_pairs * args.steps / (ms_total / 1000.0)

    # e2e: host buffers through the batch call (H2D + compute + D2H pipelined inside the library)
    eng.set_stream(0)
    eng.set_option("async", 0)
    in0 = [host[i % (nframes - 1)].data_ptr() for i in range(pairs)]
    in1 = [host[i % (nframes - 1) + 1].data_ptr() for i in range(pairs)]
    outp = [t.data_ptr() for t in out_host]

    def step_host():
        if pairs:
            eng.process_batch_ptr(in0, in1, w, h, ts, outp)

    for _ in range(2):
        step_host()
    barrier()
    cb0 = pkg.copy_bytes()
    t0 = time.perf_counter()
    each = []
    for _ in range(args.steps):
        t1 = time.perf_counter()
        step_host()  # returns when the step's results are in the host buffers
        each.append(round(1000.0 * (time.perf_counter() - t1), 2))
    torch.cuda.synchronize()
    e2e_s = reduce_max(time.perf_counter() - t0)
    cb1 = pkg.copy_bytes()
    res["clocks"] = sampler.summary()
    res["e2e"] = {"value": total_pairs * args.steps / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": int((cb1[0] - cb0[0]) // args.steps),
                  "d2h_bytes_per_step": int((cb1[1] - cb0[1]) // args.steps), "ms_each_step_this_rank": each,
                  "note": "bytes counted by the library on this rank; a frame shared by several pairs of a call is uploaded once"}
    res["out_checksum"] = int(out_host[0].to(torch.int64).sum().item()) if pairs else 0

    # ---- per-stage breakdown of one lock-step batch + the dominant kernel in the step (option "ktime": events on the lane's stream)
    burst, sustained, hbm, how = measured_peaks()
    hp, wp = (h + 31) // 32 * 32, (w + 31) // 32 * 32
    ch, cw = hp // 4, wp // 4
    fast = bool(eng.get_option("fast_active"))
    pmask = eng.get_option("plain_blocks") if fast else 0
    split = 1 if (args.precision == 1 and not (pmask & 8)) else 0  # block 3's residual chain: plain fp16 when bit 3 is set
    kb = 1
    if fast:
        kb = args.batch if args.batch > 0 else max(1, min(8, (2 * 3840 * 2176) // (hp * wp)))
        kb = min(kb, max(pairs, 1))
    stages, in_step_us = None, None
    if fast and pairs >= kb:
        eng.set_option("lanes", 1)   # (recreates the lane's runner: set before switching the stage timer on)
        eng.set_option("ktime", 1)
        nb = min(pairs, 4 * kb)
        for _ in range(3):
            eng.process_batch_ptr(d_in0[:nb], d_in1[:nb], w, h, ts[:nb], d_out[:nb], device=True)
        rep = eng.stage_report().get(0)
        eng.set_option("ktime", 0)
        eng.set_option("lanes", args.lanes)
        if rep and rep["batches"]:
            stages = {n: round(us, 1) for n, us, _ in rep["stages"]}
            if "b3 res x8" in stages:
                in_step_us = stages["b3 res x8"] / 8.0
    iters = 20
    with torch.cuda.stream(stream):
        pkg.bench_conv(stream.cuda_stream, 64, 64, ch, cw, split, 3, gpuid=local, batch=kb)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        pkg.bench_conv(stream.cuda_stream, 64, 64, ch, cw, split, iters, gpuid=local, batch=kb)
        e1.record(stream)
        torch.cuda.synchronize()
    alone_us = e0.elapsed_time(e1) / iters * 1000.0
    flop = 2.0 * 9 * 64 * 64 * ch * cw * kb  # algorithmic FLOPs per launch (SURVEY.md 3.6); a hi+lo split issues 2x this on the tensor pipe
    k_us = in_step_us if in_step_us else alone_us
    achieved = flop / (k_us * 1e-6) / 1e12
    # DRAM bytes per launch from the committed `ncu --set full` capture of this kernel (profiles/README.md)
    # keyed "<w>x<h>x<images>_<split|plain>" -> dram__bytes_read.sum + dram__bytes_write.sum of one launch
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "conv64_dram_traffic.json")))
        traffic = tj.get("%dx%dx%d_%s" % (cw, ch, kb, "split" if split else "plain"))
        if traffic is None:  # single-image capture scaled by the images per launch (the kernel re-reads nothing across images)
            one = tj.get("%dx%dx1_%s" % (cw, ch, "split" if split else "plain"))
            traffic = one * kb if one else None
    except (OSError, ValueError):
        pass
    res["roofline"] = {"bound": "tensor", "achieved": achieved, "peak": burst, "unit": "TFLOP/s", "frac": achieved / burst, "traffic": traffic,
                       "kernel": "tc_conv3x3 64->64 (+res +leaky), %d x %dx%d per launch" % (kb, cw, ch), "images_per_launch": kb,
                       "us_per_launch": k_us, "timed": "in the step: events around the 8 launches of IFBlock 3's residual chain on the lane's stream" if in_step_us else "alone",
                       "us_per_launch_alone": alone_us, "frac_alone": flop / (alone_us * 1e-6) / 1e12 / burst,
                       "peak_source": how + " bf16 burst", "tensor_issue_multiplier": 2 if split else 1,
                       "whole_model_tflops": res["value"] * GFLOP_PER_FRAME[workload] / 1000.0 if args.model == MODEL else None,
                       "whole_model_frac_of_sustained_peak": res["value"] * GFLOP_PER_FRAME[workload] / 1000.0 / sustained / world if args.model == MODEL else None}
    res["stages"] = stages
    res["fast"], res["pmask"], res["kb"] = fast, pmask, kb
    ctx.keep = (frames, host, dev, out_dev, out_host)  # freed when the next workload replaces them
    return res


def parity_block(ctx, workload, args, oracle_frame):
    """The oracle's frame for synth.pair(w, h) against the timed configuration: a full lock-step batch of that pair."""
    import numpy as np
    import parity
    w, h, _ = WORKLOADS[workload]
    a, b = parity.synth.pair(w, h)
    eng = ctx.eng
    kb = max(1, eng.get_option("batch") or max(1, min(8, (2 * 3840 * 2176) // (((h + 31) // 32 * 32) * ((w + 31) // 32 * 32)))))
    n = kb * max(1, eng.get_option("lanes"))
    outs = [np.empty_like(a) for _ in range(n)]
    eng.process_batch_ptr([a.ctypes.data] * n, [b.ctypes.data] * n, w, h, [0.5] * n, [o.ctypes.data for o in outs])
    res = parity.compare(outs[0], oracle_frame)
    res["identical_across_batch"] = bool(all(np.array_equal(outs[0], o) for o in outs[1:]))
    res["pairs_in_call"] = n
    res["oracle"] = "reference (oracle/_ref)" if parity.ref_binary() else "port (oracle/oracle_rife.cpp)"
    res["ok"] = bool(res["max_abs_diff"] <= 1 and res["psnr_db"] > 50 and res["identical_across_batch"])
    return res


def e2e_process_block(ctx, workload, args):
    """frames/s through rife_b200_process, the one call src/main.cpp:360 makes, from T caller threads on one handle."""
    import numpy as np
    import torch
    import parity
    w, h, _ = WORKLOADS[workload]
    eng = ctx.eng
    out = {}
    nf = 9
    frames = parity.synth.stream(0, nf, w, h, seed=3)
    for kind in ("pinned", "pageable"):
        if kind == "pinned":
            hold = [torch.from_numpy(f).pin_memory() for f in frames]
            ptr = [t.data_ptr() for t in hold]
        else:
            hold = [np.array(f, copy=True) for f in frames]
            ptr = [t.ctypes.data for t in hold]
        for nthreads in (1, 2, 8):
            outs = [torch.empty(h, w, 3, dtype=torch.uint8).pin_memory() if kind == "pinned" else np.empty((h, w, 3), np.uint8) for _ in range(nthreads)]
            optr = [o.data_ptr() if kind == "pinned" else o.ctypes.data for o in outs]
            calls = max(8, min(64, int(24 * nthreads ** 0.5)))
            errs = []
            gate = threading.Barrier(nthreads + 1)

            def work(t):
                try:
                    for i in range(3):  # warm-up
                        eng.process_ptr(ptr[(t + i) % (nf - 1)], ptr[(t + i) % (nf - 1) + 1], w, h, 0.5, optr[t])
                    gate.wait()
                    for i in range(calls):
                        eng.process_ptr(ptr[(t + i) % (nf - 1)], ptr[(t + i) % (nf - 1) + 1], w, h, 0.5, optr[t])
                    gate.wait()
                except Exception as e:  # pragma: no cover
                    errs.append(str(e))
                    gate.abort()

            th = [threading.Thread(target=work, args=(t,)) for t in range(nthreads)]
            for t in th:
                t.start()
            try:
                gate.wait()
                t0 = time.perf_counter()
                gate.wait()
                dt = time.perf_counter() - t0
            except threading.BrokenBarrierError:
                dt = None
            for t in th:
                t.join()
            out["%s_%dt" % (kind, nthreads)] = None if (errs or dt is None) else round(nthreads * calls / dt, 1)
    out["unit"] = "frames/s through rife_b200_process (one call per frame, H2D + compute + D2H inside each call)"
    out["combine"] = int(eng.get_option("combine"))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="1080p", choices=list(WORKLOADS), help="the headline resolution; the other one is reported under `also`")
    ap.add_argument("--only", action="store_true", help="measure only --workload (profiling runs)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--precision", type=int, default=1)
    ap.add_argument("--lanes", type=int, default=2)
    ap.add_argument("--plain-blocks", type=int, default=-1, help="bit mask of IFBlocks whose residual chain uses plain fp16 activations (-1 = library default)")
    ap.add_argument("--recompute-fm", type=int, default=-1, help="fused path: rebuild the full-resolution flow / mask planes instead of storing them (0, 1, 2; -1 = library default)")
    ap.add_argument("--head-pack", type=int, default=-1, help="fused path: packed block-head tensors (0 / 1; -1 = library default)")
    ap.add_argument("--batch", type=int, default=0, help="pairs per lock-step batch on the fused path (0 = auto from the frame size)")
    ap.add_argument("--model", default=MODEL, help="model directory name (default rife-v4.6 = the BASELINE metric; others are side measurements)")
    ap.add_argument("--tta", action="store_true")
    ap.add_argument("--tta-temporal", action="store_true")
    ap.add_argument("--timestep", type=float, default=0.5)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU leg (and with it the parity block): profiling runs only")
    ap.add_argument("--no-process-leg", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed, seeded sample of the last timed step's frames to DIR as float32 .npy (module docstring)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local)
    gpu_cpus = os.sched_getaffinity(0)  # pinned host buffers next to the GPU: the e2e legs are bound by the host link

    import torch
    import __graft_entry__ as g
    import parity
    pkg = g.load_package()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    md = parity.model_dir(args.model)
    if md is None:
        raise SystemExit("model %s not found (oracle/_ref/models or tests/models)" % args.model)
    v2, v4 = pkg.family_flags(args.model)
    eng = pkg.RIFE(local, args.tta, args.tta_temporal, False, 1, v2, v4)
    # weights: rank 0 reads the model directory, everyone else receives the packed blob over NCCL (NVLink)
    if world > 1:
        sys.path.insert(0, os.path.join(ROOT, "rife-ncnn-vulkan_b200"))
        import dist_util
        blob = None
        if rank == 0:
            eng.load(md)
            blob = eng.export_weights()
        blob = dist_util.broadcast_blob(blob, dist, device=torch.device("cuda", local))
        if rank != 0:
            eng.load_packed(blob)
    else:
        eng.load(md)
    eng.set_option("precision", args.precision)
    eng.set_option("lanes", args.lanes)
    eng.set_option("batch", args.batch)
    if args.plain_blocks >= 0:
        eng.set_option("plain_blocks", args.plain_blocks)
    if args.recompute_fm >= 0:
        eng.set_option("recompute_fm", args.recompute_fm)
    if args.head_pack >= 0:
        eng.set_option("head_pack", args.head_pack)

    ctx = Ctx()
    ctx.pkg, ctx.eng, ctx.dist, ctx.world, ctx.rank, ctx.local = pkg, eng, dist, world, rank, local
    ctx.l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    ctx.stream = torch.cuda.Stream()
    link = host_link_gbs() if rank == 0 else None

    order = [args.workload] + ([] if args.only else [k for k in WORKLOADS if k != args.workload])
    results, rc = {}, 0
    plain_v46 = args.model == MODEL and not (args.tta or args.tta_temporal)
    for wl in order:
        r = measure(ctx, wl, args, wl == args.workload)
        if rank == 0:
            r["cpu_baseline"], r["parity"] = None, None
            if not args.no_cpu_baseline and plain_v46:
                os.sched_setaffinity(0, all_cpus)  # the CPU leg may use every host core
                try:
                    cpu, frame = cpu_reference(wl, 2 if wl == "1080p" else 1, threads=results[order[0]]["cpu_baseline"]["cores"] if (results and results[order[0]].get("cpu_baseline") and results[order[0]]["cpu_baseline"].get("cores")) else None)
                    r["cpu_baseline"] = cpu
                    r["parity"] = parity_block(ctx, wl, args, frame)
                    if not r["parity"]["ok"]:
                        rc = 3
                except Exception as e:  # the oracle binary did not travel / wrong ISA: report, do not fake
                    r["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": 0, "kind": "unavailable", "sample": str(e)[:200]}
            os.sched_setaffinity(0, gpu_cpus)  # back next to the GPU for the remaining host-buffer legs
            if world == 1 and not args.no_process_leg and plain_v46:
                r["e2e_process"] = e2e_process_block(ctx, wl, args)
        results[wl] = r
        if dist is not None:
            dist.barrier()

    if rank == 0:
        def block(wl):
            r = results[wl]
            _, _, desc = WORKLOADS[wl]
            b = {"value": r["value"], "unit": "frames/s", "ms_per_step": r["ms_per_step"], "pairs_per_step": r["pairs_per_step_all_ranks"], "e2e": r["e2e"],
                 "gpu_launches": r["gpu_launches"], "clocks": r["clocks"], "roofline": r["roofline"], "stages_us_per_lockstep_batch": r["stages"],
                 "parity": r.get("parity"), "cpu_baseline": r.get("cpu_baseline"), "e2e_process": r.get("e2e_process"),
                 "gflop_per_frame": GFLOP_PER_FRAME[wl] if plain_v46 else None, "out_checksum": r["out_checksum"], "workload": desc}
            return b
        head = results[args.workload]
        w, h, desc = WORKLOADS[args.workload]
        pmask = head["pmask"]
        hb = block(args.workload)
        line = {"metric": "interpolated frames/sec (%s)" % args.model, "value": hb["value"], "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": hb["ms_per_step"], "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": ("f16 operands / f32 accumulate (split hi+lo operands in block heads%s)" % ("" if pmask == 15 else " and IFBlocks " + ",".join(str(k) for k in range(4) if not (pmask >> k) & 1)))
                         if args.precision == 1 else ("f32" if args.precision == 0 else "f16 / f32 accumulate"),
                "data": "synthetic",
                "config": {"workload": desc if args.model == MODEL else desc.replace("rife-v4.6", args.model), "timestep": args.timestep, "tta": args.tta,
                           "tta_temporal": args.tta_temporal, "pairs_per_step": head["pairs_per_step_all_ranks"], "precision_tier": args.precision, "lanes": args.lanes, "batch": args.batch,
                           "images_per_lockstep_batch": head["kb"], "plain_fp16_blocks_mask": eng.get_option("plain_blocks"), "recompute_fm": eng.get_option("recompute_fm"), "head_pack": eng.get_option("head_pack"),
                           "wide_tiles": int(os.environ.get("RIFE_B200_WIDE", "0")),  # library default TC_WIDE_DEFAULT = 0 (csrc/tc_conv.h)
                           "fused_path": head["fast"], "l2": "flushed between timed steps (256 MiB memset)", "weights": "reference model files" if "_ref" in md else "synthetic",
                           "host_numa": numa, "host_link_GBps": link},
                "gflop_per_frame": hb["gflop_per_frame"], "model_tflops": hb["value"] * GFLOP_PER_FRAME[args.workload] / 1000.0 if plain_v46 else None,
                "e2e": hb["e2e"], "e2e_process": hb["e2e_process"], "gpu_launches": hb["gpu_launches"], "clocks": hb["clocks"], "roofline": hb["roofline"],
                "stages_us_per_lockstep_batch": hb["stages_us_per_lockstep_batch"], "parity": hb["parity"], "cpu_baseline": hb["cpu_baseline"], "out_checksum": hb["out_checksum"],
                "also": {wl: block(wl) for wl in order[1:]}}
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return rc


if __name__ == "__main__":
    sys.exit(main())
