#!/usr/bin/env python
"""bench.py - IQ Msamples/s of the composite-video -> IQ hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]

A *step* is one pass of the hot path over one batch: FRAMES video frames (default 1024 =
640 000 scan lines = 655 M complex samples, rendered in 16 calls of 64 frames = 164 MB of
int16 IQ each - larger than the 126 MB L2 - into the same device buffer; 20 steps keep the
GPU busy for > 100 ms, so the 1 kHz clock sampler sees the timed region) of BASELINE config 2: PAL System I, 16 Msps, --filter (VSB) + FM mono + NICAM-728 +
colour, built-in test pattern and tone. With N GPUs each rank renders its own independent
RF channel on its own GPU (weak scaling, no collective on the data path); `value` is
the sum over channels divided by the slowest rank's device time.

Keys beyond the base contract:
  roofline      HBM-write roofline of the dominant kernel (k_line, the fused line kernel):
                algorithmic bytes (4 B per complex sample) / CUDA-event duration of that
                kernel, vs the measured copy bandwidth in MEASURED_PEAKS.json; step_frac is
                the same for the whole step, issue the kernel's issue-slot figures from ncu.
  extra         device-resident lines for the other BASELINE configs (1, 3, 4, 5) and, at
                N = 1, the drop-in path: hacktv's own CLI on the adapter vs the stock CLI.
  e2e           the same metric through htv_render_host() with HOST buffers: every
                step uploads its pictures (a live source: one upload per frame) and sound,
                renders, and copies the IQ back to pinned host memory.
  cpu_baseline  the UNMODIFIED reference (oracle/_ref/ref_harness) timed on this box's
                host cores on a bounded sample of the same workload (rank 0, N = 1 only).

--impl reference times the reference's own CPU implementation with every host thread it
can use (as many concurrent encoder instances as fit; one instance = 1 + nthreads
pthreads) and prints the same JSON line with "impl": "reference".

--dump-outputs DIR writes what the last timed step computed, as float32 arrays of whole
lines of int16 IQ (I, Q interleaved; rows in stream order): DIR/iq.npy from the
device-resident step, a fixed seeded choice of lines of each of its render calls, gathered on
the device after each call of that step; DIR/e2e_iq.npy a seeded choice of lines of the host
buffer of the last end-to-end step. 60 MB at most in all. The inputs (test pattern and tone) are the
same on every run, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODE, RATE, FILTER = "i", 16_000_000, True
WORKLOAD = "PAL-I (-m i) 16 Msps --filter: VSB + FM mono + NICAM-728 + colour, built-in test pattern"
WORKLOADS = {   # --workload: the metric is quoted on cfg2; cfg5 is BASELINE config 5's per-channel load (20 Msps)
    "cfg2": ("i", 16_000_000, True, WORKLOAD),
    "cfg5": ("i", 20_000_000, True, "PAL-I (-m i) 20 Msps --filter: VSB + FM mono + NICAM-728 + colour, built-in test pattern (BASELINE config 5, per channel)"),
}
CHUNK_FRAMES = 64        # frames per htv_render call: 164 MB of IQ at 16 Msps, larger than the L2
REF_HARNESS = os.path.join(ROOT, "oracle", "_ref", "ref_harness")
REF_THREADS = 3          # main/raster + vfilter + audio (reference video.c:4692: 1 + nthreads)
# From the ncu --set full capture of the shipped k_line (profiles/r02_summary.md), per scan line of 1024 samples:
# dram__bytes_read.sum + dram__bytes_write.sum of one launch over 40 000 lines, and the issue-slot figures.
NCU = {"file": "profiles/r02_ncu_k_line_raw.txt", "lines": 40000, "dram_read": 47_632_128, "dram_write": 113_646_080,
       "warp_instructions": 238_153_871, "issue_active_pct": 61.8}
KERNEL = "k_line (fused line kernel: raster + chroma and video filters on the tensor cores + sound carriers + IQ store)"
DUMP_BYTES = {"iq": 45_000_000, "e2e_iq": 15_000_000}     # --dump-outputs: float32 bytes per array


def dump_lines(lines, calls, values_per_line, nbytes):
    """--dump-outputs: for each of `calls` render calls of `lines` lines, a sorted choice of its lines, as many
    as fit `nbytes` of float32 over all calls; seeded, so the same on every run."""
    k = max(1, min(lines, nbytes // 4 // values_per_line // calls))
    rng = np.random.default_rng(0)
    return np.stack([np.sort(rng.choice(lines, k, replace=False)) for _ in range(calls)])


def save_dump(directory, name, rows):
    np.save(os.path.join(directory, name + ".npy"), rows.reshape(-1, rows.shape[-1]).astype(np.float32))


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md) through
    NVML at ~1 kHz (the region is only milliseconds long; spawning nvidia-smi is too slow).
    Falls back to one nvidia-smi query if NVML is unavailable."""

    def __init__(self, index):
        self.index, self.rows, self._stop = index, [], threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)
        self.t0 = self.t1 = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            # torch device index -> NVML handle (respects CUDA_VISIBLE_DEVICES through the UUID)
            import torch
            uuid = str(torch.cuda.get_device_properties(index).uuid)
            try:
                self._h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._max = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                if nv:
                    clk = nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                    self.rows.append((time.perf_counter(), clk, self._max, rs))
                else:
                    q = "clocks.sm,clocks.max.sm"
                    r = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                       capture_output=True, text=True, timeout=5)
                    p = [x.strip() for x in r.stdout.strip().split(",")]
                    self.rows.append((time.perf_counter(), int(p[0]), int(p[1]), 0))
            except Exception:
                pass
            self._stop.wait(0.001 if nv else 0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=3)

    def summary(self):
        rows = [r for r in self.rows if self.t0 is None or (self.t0 <= r[0] <= self.t1)] or self.rows
        sm = sorted(r[1] for r in rows)
        reasons = set()
        nv = self._nv
        if nv:
            names = {"hw_slowdown": "nvmlClocksEventReasonHwSlowdown", "hw_thermal_slowdown": "nvmlClocksEventReasonHwThermalSlowdown",
                     "sw_thermal_slowdown": "nvmlClocksEventReasonSwThermalSlowdown", "sw_power_cap": "nvmlClocksEventReasonSwPowerCap"}
            for r in rows:
                for k, attr in names.items():
                    bit = getattr(nv, attr, None) or getattr(nv, attr.replace("Event", "Throttle"), 0)
                    if bit and (r[3] & bit):
                        reasons.add(k)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max((r[2] for r in rows), default=None),
                "reasons": sorted(reasons), "samples": len(rows), "source": "nvml" if nv else "nvidia-smi"}


def cpu_budget():
    """Host threads this process may really use: the affinity mask, capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(int(quota) // int(period))))
    except Exception:
        pass
    return n


def run_reference_instances(ninst, frames, timeout=900, mode=MODE, rate=RATE, filt=FILTER):
    """ninst concurrent reference encoders, each timing `frames` frames after a 2-frame
    warm-up; returns (aggregate Msamples/s, per-instance list, wall seconds)."""
    lines = frames * 625
    cmd = ["timeout", str(timeout), REF_HARNESS, "-m", mode, "-s", str(rate), "--skip", "1250", "--lines", str(lines), "--bench"]
    if filt:
        cmd.append("--filter")
    t0 = time.time()
    procs = [subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True) for _ in range(ninst)]
    outs = [p.communicate()[0] for p in procs]
    wall = time.time() - t0
    per = []
    for o in outs:
        for ln in o.splitlines():
            if ln.startswith("{") and "msamples_per_s" in ln:
                per.append(json.loads(ln)["msamples_per_s"])
    if len(per) != ninst:
        raise RuntimeError("reference harness failed")
    return sum(per), per, wall


def bench_reference(args, rank, world):
    if rank != 0:
        return
    mode, rate, filt, workload = WORKLOADS[args.workload]
    cores = cpu_budget()
    if not os.path.exists(REF_HARNESS):
        emit({"impl": "reference", "unavailable": "oracle/_ref/ref_harness was not built (no reference tree at build time)"})
        return
    # one reference encoder = main + video-filter + audio thread and cannot use more: as many encoders as fit the
    # threads this process may use (affinity mask and cgroup quota, not the machine's core count)
    ninst = max(1, cores // REF_THREADS)
    frames = args.ref_frames
    single, _, _ = run_reference_instances(1, max(25, frames // 2), mode=mode, rate=rate, filt=filt)
    for _ in range(args.warmup):
        run_reference_instances(ninst, max(2, frames // 4), mode=mode, rate=rate, filt=filt)
    vals, t, pers = [], 0.0, []
    for _ in range(args.steps):
        agg, per, wall = run_reference_instances(ninst, frames, mode=mode, rate=rate, filt=filt)
        vals.append(agg)
        pers += per
        t += wall
    v = sum(vals) / len(vals)
    pers.sort()
    sample = f"{ninst} concurrent reference encoders x {frames} frames ({frames * 625 * (rate // 15625) / 1e6:.1f} Msamples each) per step, vid_next_line loop, no sink I/O"
    emit({
        "impl": "reference", "metric": "IQ Msamples/s", "value": round(v, 3), "unit": "Msamples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(1000 * t / args.steps, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int16 (int32/int64 accumulate)", "data": "synthetic",
        "config": {"workload": workload, "parallelism": f"{ninst} processes x {REF_THREADS} threads on {cores} usable host threads ({os.cpu_count()} in the machine)"},
        "cpu_baseline": {"value": round(v, 3), "unit": "Msamples/s", "cores": ninst * REF_THREADS, "kind": "reference", "sample": sample,
                         "per_instance_msamples_per_s": {"min": round(pers[0], 2), "median": round(pers[len(pers) // 2], 2), "max": round(pers[-1], 2)},
                         "single_encoder_alone_msamples_per_s": round(single, 2)},
        "e2e": {"value": round(v, 3), "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


def channel_of_rank(rank, world, nchannels):
    """Whole RF channels are the unit of parallelism (SURVEY.md section 8e): channel c belongs to rank c mod world."""
    return [c for c in range(nchannels) if c % world == rank]


def reduce_job(torch, dist, world, ms, samples, device="cuda"):
    """What the ranks exchange - and all they exchange: the slowest rank's device time (MAX) and the samples every
    rank rendered (SUM). Returns (ms of the job, samples of the job)."""
    t = torch.tensor([float(ms), float(samples)], dtype=torch.float64, device=device)
    if world > 1:
        tm, ts = t[:1].clone(), t[1:].clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        return tm.item(), ts.item()
    return t[0].item(), t[1].item()


def bind_to_gpu_numa(local):
    """Pin this rank to the host cores next to its GPU (NVML's CPU affinity of the device) BEFORE any pinned
    memory is allocated: with 8 ranks on a two-socket box the staging buffers and the copy threads of GPUs 4-7
    otherwise land on the far socket (round 1: e2e scaling 0.76 at N = 8)."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(local).uuid)
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w in range(words) for b in range(64) if (int(mask[w]) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def prefer_gpu_memory_node(local):
    """Pinned staging buffers on the NUMA node the GPU hangs off (sysfs numa_node of its PCI function), by a
    MPOL_PREFERRED memory policy set before anything is allocated: DMA that crosses the socket link costs duplex
    bandwidth. Returns what was found and done, for the e2e record; never raises."""
    info = {}
    try:
        import ctypes
        import torch
        p = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (getattr(p, "pci_domain_id", 0), p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        info["gpu_numa_node"] = node
        try:
            with open("/sys/devices/system/node/online") as f:
                info["nodes_online"] = f.read().strip()
        except OSError:
            pass
        import platform
        if node >= 0 and platform.machine() == "x86_64":              # the syscall number below is x86-64's
            mask = (ctypes.c_ulong * 16)()
            mask[node // 64] = 1 << (node % 64)
            libc = ctypes.CDLL(None, use_errno=True)
            r = libc.syscall(238, 1, ctypes.byref(mask), 1024)          # set_mempolicy(MPOL_PREFERRED, mask, maxnode)
            info["mempolicy"] = "preferred node %d" % node if r == 0 else "set_mempolicy errno %d" % ctypes.get_errno()
    except Exception as e:                                                # sysfs not there, not x86-64, ...
        info["note"] = type(e).__name__
    return info


def device_resident(H, torch, mode, rate, filt, frames, steps, warmup, stream, clock_index=None, **kw):
    """K steps of `frames` frames each, rendered in calls of CHUNK_FRAMES into one device buffer; CUDA events."""
    enc = H.Encoder(H.mode_config(mode, vfilter=filt, **kw), rate)
    enc.open_test_source()
    chunk = min(frames, CHUNK_FRAMES) * enc.lines
    calls = max(1, frames // min(frames, CHUNK_FRAMES))
    nsamp = chunk * enc.width
    out = torch.empty(nsamp * (2 if enc.complex else 1), dtype=torch.int16, device="cuda")
    enc.set_kernel_timing(True)
    for _ in range(warmup):
        enc.render(chunk, out.data_ptr(), stream)
    torch.cuda.synchronize()
    l0 = enc.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    return enc, out, chunk, calls, nsamp, l0, ev0, ev1


def quick_config(H, torch, stream, name, mode, rate, filt, frames=CHUNK_FRAMES, iters=10):
    """One device-resident line for a BASELINE config that is not the metric's workload (for `extra`)."""
    enc = H.Encoder(H.mode_config(mode, vfilter=filt), rate)
    enc.open_test_source()
    n = frames * enc.lines
    out = torch.empty(n * enc.width * (2 if enc.complex else 1), dtype=torch.int16, device="cuda")
    for _ in range(3):
        enc.render(n, out.data_ptr(), stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        enc.render(n, out.data_ptr(), stream)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    msps = n * enc.width / (ms / 1e3) / 1e6
    enc.close()
    return {"config": name, "frames_per_step": frames, "ms_per_step": round(ms, 4), "msamples_per_s": round(msps, 1),
            "realtime_x": round(msps / (rate / 1e6), 1)}


def dropin_throughput(seconds=4.0):
    """The path a hacktv user runs: hacktv's own CLI (-o file sink) on the adapter (integration/video_b200.c:
    vid_next_line over the prefetching frame pipeline + rf_write) against the stock binary, same command line."""
    dropin = os.path.join(ROOT, "oracle", "_ref", "hacktv_b200_dropin")
    stock = os.path.join(ROOT, "oracle", "_ref", "hacktv_ref")
    if not (os.path.exists(dropin) and os.path.exists(stock)):
        return None
    args = ["-m", "i", "-s", "16000000", "--filter"]
    out = {"command": "-m i -s 16000000 --filter -o <sink> test"}

    def piped(binary, nsamples):
        """-o - into a pipe that is read and dropped: time for nsamples complex samples"""
        t0 = time.time()
        cmd = f"HACKTV_B200_PREFETCH=1 timeout 120 {binary} {' '.join(args)} -o - test 2>/dev/null | head -c {nsamples * 4} | wc -c"
        r = subprocess.run(["bash", "-c", cmd], capture_output=True, text=True)
        dt = time.time() - t0
        got = int((r.stdout.strip() or "0").split()[-1])
        return round(got / 4 / dt / 1e6, 1) if got else None

    # the stock encoder: ~60 Msamples/s, 2 s of signal through a pipe costs nothing extra
    out["stock"] = {"msamples_per_s_pipe": piped(stock, 32_000_000)}
    # the adapter: the same pipe (what `hacktv -o - | consumer` delivers: bounded by the 64 KB pipe), and the file
    # sink proper (-o /dev/null), timed inside the adapter (HACKTV_STATS: lines / seconds between the first
    # vid_next_line and vid_free)
    out["b200"] = {"msamples_per_s_pipe": piped(dropin, 256_000_000)}
    p = subprocess.Popen(["timeout", "-s", "INT", str(seconds), dropin] + args + ["-o", "/dev/null", "test"],
                         stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, env=dict(os.environ, HACKTV_STATS="1", HACKTV_B200_PREFETCH="1"))
    err = p.communicate()[1]
    for ln in err.splitlines():
        if ln.startswith("{") and "lines" in ln:
            st = json.loads(ln)
            out["b200"]["msamples_per_s_file_sink"] = round(st["lines"] * 1024 / st["seconds"] / 1e6, 1)
            out["b200"]["seconds"] = round(st["seconds"], 2)
    if out["stock"]["msamples_per_s_pipe"]:
        best = out["b200"].get("msamples_per_s_file_sink") or out["b200"]["msamples_per_s_pipe"]
        if best:
            out["speedup_vs_stock_cli"] = round(best / out["stock"]["msamples_per_s_pipe"], 1)
    return out


_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version line at the first
    collective when NCCL_DEBUG=VERSION): everything but the result goes to stderr."""
    global _STDOUT
    sys.stdout.flush()
    _STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(obj):
    sys.stdout.flush()
    if _STDOUT is not None:
        os.dup2(_STDOUT, 1)
    print(json.dumps(obj), flush=True)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--frames", type=int, default=1024, help="video frames per step (rendered in calls of 64 frames)")
    ap.add_argument("--e2e-frames", type=int, default=64, help="video frames per end-to-end step")
    ap.add_argument("--ref-frames", type=int, default=100, help="frames per reference instance per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        bench_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import hacktv_b200 as H

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    numa_cpus = bind_to_gpu_numa(local)
    numa_mem = prefer_gpu_memory_node(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    mode, rate, filt, workload = WORKLOADS[args.workload]
    conf = H.mode_config(mode, vfilter=filt)
    stream = torch.cuda.current_stream().cuda_stream

    # ---- device-resident throughput ("value") ---------------------------------
    enc, out, chunk, calls, nsamp, l0, ev0, ev1 = device_resident(H, torch, mode, rate, filt, args.frames, args.steps, args.warmup, stream)
    nlines = chunk * calls
    dump = args.dump_outputs if rank == 0 else None
    picked = None
    if dump:
        os.makedirs(dump, exist_ok=True)
        out_lines = out.view(chunk, -1)
        pick = torch.from_numpy(dump_lines(chunk, calls, out_lines.shape[1], DUMP_BYTES["iq"])).cuda()
        picked = torch.empty((calls, pick.shape[1], out_lines.shape[1]), dtype=torch.int16, device="cuda")
        torch.index_select(out_lines, 0, pick[0], out=picked[0])       # its first launch loads the kernel: not timed
    barrier()
    with ClockSampler(local) as clk:
        time.sleep(0.005)
        clk.t0 = time.perf_counter()
        ev0.record()
        for step in range(args.steps):
            for c in range(calls):
                enc.render(chunk, out.data_ptr(), stream)
                if picked is not None and step == args.steps - 1:      # the next call overwrites `out`
                    torch.index_select(out_lines, 0, pick[c], out=picked[c])
        ev1.record()
        barrier()
        clk.t1 = time.perf_counter()
    ms = ev0.elapsed_time(ev1)
    launches = enc.kernel_launches - l0
    clocks = clk.summary()
    # per-launch duration of the dominant kernel, CUDA events on its own stream (untimed extra steps)
    kern_ms = []
    for _ in range(3):
        enc.render(chunk, out.data_ptr(), stream)
        torch.cuda.synchronize()
        kern_ms.append(enc.last_line_kernel_ms())
    kern_lines = enc.last_line_kernel_lines()
    checksum = int(out[:4096].to(torch.int32).sum().item())
    if picked is not None:
        save_dump(dump, "iq", picked.cpu().numpy())
    width = enc.width
    enc.close()
    del out

    # ---- end to end through the C-ABI with host buffers ("e2e") -----------------
    e2e = None
    if not args.no_e2e:
        e2e_frames = args.e2e_frames
        enc2 = H.Encoder(conf, rate)
        e2e_lines = e2e_frames * enc2.lines
        # a live source: a ring of 8 pinned capture buffers, a new picture (serial) every frame -> every frame is
        # uploaded; frames that follow each other in the ring go up in one copy
        one = H.test_pattern(enc2.active_width, enc2.active_lines).astype(np.int32)
        pic = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(one, (8,) + one.shape))).pin_memory()
        tone = torch.from_numpy(H.test_tone()).pin_memory()
        enc2.open_memory_source(pic.numpy().view(np.uint32), tone.numpy(), audio_block=8192, static_video=False)
        host = torch.empty(e2e_lines * enc2.width * 2, dtype=torch.int16).pin_memory()
        for _ in range(max(1, args.warmup)):
            enc2.render_host_ptr(e2e_lines, host.data_ptr())
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            enc2.render_host_ptr(e2e_lines, host.data_ptr())
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if dump:
            per = 2 if enc2.complex else 1
            rows = host[: e2e_lines * enc2.width * per].view(e2e_lines, -1).numpy()
            save_dump(dump, "e2e_iq", rows[dump_lines(e2e_lines, 1, rows.shape[1], DUMP_BYTES["e2e_iq"])])
        e2e_samples = e2e_lines * enc2.width
        e2e_s, e2e_job = reduce_job(torch, dist, world, dt, e2e_samples * args.steps)
        h2d = e2e_frames * enc2.active_width * enc2.active_lines * 4 + int(e2e_samples / rate * 32000) * 4
        e2e = {"value": round(e2e_job / e2e_s / 1e6, 2), "unit": "Msamples/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": e2e_samples * 4,
               "frames_per_step": e2e_frames, "ms_per_step": round(1000 * e2e_s / args.steps, 3),
               "checksum": int(host[:4096].to(torch.int32).sum().item()),
               "api": "htv_av_memory_open (ring of 8 pinned pictures, every frame uploaded) + htv_render_host (C-ABI), pinned host buffers",
               "numa_bound_cpus": numa_cpus, "numa_memory": numa_mem}
        enc2.close()

    step_samples = nlines * width
    ms_max, job_samples = reduce_job(torch, dist, world, ms, step_samples * args.steps)

    if rank == 0:
        value = job_samples / (ms_max / 1e3) / 1e6
        peak, peak_src = measured_peak_gbs()
        k_ms = sorted(kern_ms)[len(kern_ms) // 2]
        k_samples = kern_lines * width
        achieved = k_samples * 4 / (k_ms / 1e3) / 1e9 if k_ms > 0 else None
        step_gbs = step_samples * 4 * args.steps / (ms_max / 1e3) / 1e9      # per GPU: every rank writes its own IQ
        cpu = None
        if world == 1 and not args.no_cpu_baseline and os.path.exists(REF_HARNESS):
            v, per, wall = run_reference_instances(1, 150, mode=mode, rate=rate, filt=filt)
            cpu = {"value": round(v, 3), "unit": "Msamples/s", "cores": REF_THREADS, "kind": "reference",
                   "sample": "1 reference encoder (main + vfilter + audio threads), 150 frames after a 2-frame warm-up, "
                             "vid_next_line loop, no sink I/O (oracle/_ref/ref_harness)",
                   "host_cores": os.cpu_count(), "usable_host_threads": cpu_budget()}
        extra = None
        if world == 1 and not args.no_extra:
            extra = {"configs": [
                quick_config(H, torch, stream, "cfg1: -m pal -s 16000000 (baseband, real int16)", "pal", 16_000_000, False),
                quick_config(H, torch, stream, "cfg3: -m m -s 13500000 --filter", "m", 13_500_000, True),
                quick_config(H, torch, stream, "cfg4: -m l -s 16000000 --filter (SECAM)", "l", 16_000_000, True),
                quick_config(H, torch, stream, "cfg5 (one channel): -m i -s 20000000 --filter", "i", 20_000_000, True)],
                "dropin_cli": dropin_throughput()}
        per_line = 1.0 / NCU["lines"]
        emit({
            "metric": "IQ Msamples/s", "value": round(value, 2), "unit": "Msamples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_max / args.steps, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int16 (int32 accumulate; RGB->YUV table built in fp64 at init)", "data": "synthetic",
            "config": {"workload": workload, "frames_per_step": calls * min(args.frames, CHUNK_FRAMES), "lines_per_step": nlines,
                       "calls_per_step": calls, "frames_per_call": min(args.frames, CHUNK_FRAMES),
                       "samples_per_step_per_gpu": step_samples, "parallelism": f"{world} independent RF channel(s), one per GPU, no collectives",
                       "l2": f"every call writes {nsamp * 4 / 1e6:.0f} MB of IQ per GPU (> 126 MB L2); tables are L2-resident by design",
                       "ms_per_64_frames": round(ms_max / args.steps / calls, 4),
                       "realtime_x": round(value / world / (rate / 1e6), 1)},
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1) if achieved else None, "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4) if achieved else None,
                         "traffic": int(round((NCU["dram_read"] + NCU["dram_write"]) * per_line * kern_lines)) if width == 1024 else None,
                         "kernel": KERNEL, "kernel_ms": round(k_ms, 4),
                         "lines_per_launch": kern_lines, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": k_samples * 4,
                         "step_achieved": round(step_gbs, 1), "step_frac": round(step_gbs / peak, 4),
                         "issue": {"slots_per_sample": round(NCU["warp_instructions"] * 32 / (NCU["lines"] * 1024), 1),
                                   "issue_active_pct": NCU["issue_active_pct"], "source": NCU["file"]},
                         "note": "4 B per complex sample written once; the kernel is issue-slot bound (DESIGN.md section 4), not HBM bound"},
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "checksum": checksum,
            "extra": extra,
        })

    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
