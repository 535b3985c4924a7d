#!/usr/bin/env python
"""bench.py — Msamples/s through iq_tool's resample+shift+filter chain on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2] [--dump-outputs DIR]

A "step" is one pass of the whole hot path (convert -> DC block -> multi-stage resample -> FIR ->
convert) over one HBM-resident synthetic capture of the workload BASELINE.json's metric is
quoted on (configs[1] = cfg2: cs16 @ 20 Msps -> 744187.5 sps, 255-tap low-pass FIR + DC block).
With N > 1 (torchrun, one rank per GPU) the capture is time-sharded: rank r owns input frames
[r*n, (r+1)*n) of an N*n-frame capture, re-computes a filter/DC halo in front of its shard and
no collective touches the data path (weak scaling).

Prints ONE JSON line (see the task contract): value = whole-job Msamples/s with inputs resident
in HBM, e2e = the same metric through the host-buffer C-ABI call (pinned host memory, H2D + D2H
inside the timed region), roofline = the dominant kernel against the measured HBM peak, and
cpu_baseline = the reference's stage code (oracle/_ref, on the restated liquid layer) timed on
the host cores for a bounded sample.
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

METRIC = "Msamples/s through resample+shift+filter chain"
UNIT = "Msamples/s"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", d
    return 6650.0, "fallback (B200_PROFILING.md)", {}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.lines = []
        self.proc = None
        self.t = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def rd():
            for ln in self.proc.stdout:
                self.lines.append((time.time(), ln.strip()))
        self.t = threading.Thread(target=rd, daemon=True)
        self.t.start()

    def stop(self, t0: float, t1: float):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []                                  # (timestamp, sm clock, max clock, power, reasons)
        for ts, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mx = float(f[1]), float(f[2])
            except ValueError:
                continue
            if clk <= 0:
                continue
            try:
                pw = float(f[3])
            except ValueError:
                pw = None
            rows.append((ts, clk, mx, pw, {nm for k, nm in enumerate(names) if f[5 + k].lower().startswith("active")}))
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no nvidia-smi samples"]}
        inside = [r for r in rows if t0 - 0.03 <= r[0] <= t1 + 0.03]
        note = None
        if not inside:
            # timed region shorter than the sampling period: the samples nearest to it (the sampler runs from before the
            # warm-up steps, so these are still samples under load)
            mid = 0.5 * (t0 + t1)
            inside = sorted(rows, key=lambda r: abs(r[0] - mid))[:3]
            note = "timed region shorter than the sampling period: nearest samples"
        reasons = set().union(*[r[4] for r in inside])
        power = [r[3] for r in inside if r[3] is not None]
        out = {"sm_mhz": statistics.median([r[1] for r in inside]), "sm_max_mhz": rows[-1][2], "reasons": sorted(reasons),
               "samples": len(inside), "power_w_max": max(power) if power else None}
        if note:
            out["note"] = note
        return out


def dc_local_state(cfg, info):
    """DC blocker evaluated with a local state per warp stretch (no pre-pass over the input; a closed-form correction pass
    over the resampled stream instead)."""
    return bool(cfg.dc_block and not cfg.iq_correction and not (cfg.freq_shift_hz and not cfg.shift_after_resample)
                and info.fused_front)


# ALGORITHMIC bytes per INPUT sample for each kernel class of a workload (SURVEY 8(d) / DESIGN.md Kernels): what an ideal
# implementation must move.  Passes an implementation adds on top (the DC correction pass of the fused front: 16 r) show up
# in `traffic` and in the time, never here.
def class_bytes_per_sample(cfg, info):
    r = info.ratio
    inb, outb = cfg.in_bytes, cfg.out_bytes
    return {
        "fused_front": inb + 8.0 * r,          # raw in, resampled cf32 out
        "pre": inb + 8.0,                      # raw in, cf32 out
        "dc_scan": float(inb),                 # raw in
        "resampler": 8.0 + 8.0 * r,            # cf32 in, cf32 out (ideal, no inter-stage traffic)
        "filter": 16.0 * r,                    # cf32 in/out at the output rate
        "post": (8.0 + outb) * r,
    }


def chain_flops_per_sample(cfg, info):
    """FP32 FLOPs (FMA = 2) per input sample actually required by the chain (DESIGN.md)."""
    fl = 2.0  # convert
    if cfg.dc_block:
        fl += 6.0
    if cfg.freq_shift_hz and not cfg.shift_after_resample:
        fl += 6.0
    S = info.num_halfband
    rate = 1.0
    for d in range(S):
        m = info.halfband_m[S - 1 - d]
        rate *= 0.5
        fl += rate * (8.0 * m + 2.0)
    fl += info.ratio * 56.0
    if info.filter_num_taps and info.filter_impl in (3, 4):     # FFT block filter: 2 transforms of 2n per n outputs
        import math
        fl += info.ratio * (20.0 * math.log2(2.0 * max(1, info.filter_block_size)) + 12.0)
    elif info.filter_num_taps:
        fl += info.ratio * info.filter_num_taps * (8.0 if info.filter_impl == 2 else 4.0)
    fl += info.ratio * 4.0
    return fl


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (its stage sources
    compiled in place, oracle/_ref) with the reference's thread model (one thread per stage),
    on a bounded sample of the same workload per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import numpy as np
    from iq_tool_b200 import baseline_workloads
    from iq_tool_b200.synth import synth_numpy
    from oracle.loader import CpuChain, have_ref
    wl = baseline_workloads()[args.workload.split(":", 1)[-1]]      # file:<cfg> times the same chain
    kind = "ref_fast" if have_ref(fast=True) else "oracle"
    # bounded sample: about 25 s of CPU work for the whole run whatever --steps is (the CPU chain does ~50 Msamples/s)
    n = min(args.cpu_samples, max(1 << 20, int(1.25e9 / max(1, args.steps))))
    n -= n % 16384
    raw = synth_numpy(wl, n)
    ch = CpuChain(wl.config, kind)
    threaded = kind != "oracle"
    for _ in range(args.warmup):
        ch.process(raw[: 2 * min(n, 1 << 20)], threaded=threaded)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = ch.process(raw, threaded=threaded)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out.view(np.uint8).reshape(-1, wl.config.out_bytes), wl.config.output_format)
    val = n * args.steps / dt / 1e6
    cores = 3 if threaded else 1
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{wl.name}: {wl.description}", "frames_per_step": n},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores,
                         "kind": "reference" if kind != "oracle" else "port",
                         "sample": f"{n} input frames per step; reference stage sources (-O3 -ffast-math) on the "
                                   f"restated liquid layer (SCALAR dot products: a floor for a real AVX libliquid, not its "
                                   f"speed), pre/resampler/post stage threads as in pipeline.c:99-116"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "host_cpus": os.cpu_count(),
    }
    print(json.dumps(line))
    return 0


class WorkloadRun:
    """One workload on this rank: the HBM-resident capture (one time shard of it when world > 1), the chain, and the
    step the bench times — `restart` (or closed-form seek to the shard lead) + one device-resident pass over the capture."""

    def __init__(self, name, args, world, rank, local_rank, dev, stream, samples=0):
        import torch
        from iq_tool_b200 import baseline_workloads, gpu
        from iq_tool_b200.configs import stage_workloads
        from iq_tool_b200.shard import ShardedChain
        from iq_tool_b200.synth import synth_torch
        self.gpu, self.torch = gpu, torch
        self.args, self.world, self.rank, self.local_rank, self.dev, self.stream = args, world, rank, local_rank, dev, stream
        self.wl = {**baseline_workloads(), **stage_workloads()}[name]
        self.cfg = self.wl.config
        n = samples or self.wl.throughput_samples
        self.n = n - n % 16384
        # N > 1: the capture of world*n frames is time-sharded (iq_tool_b200/shard.py): closed-form seek, halo in front of
        # the shard, and — for digital-AGC chains — the per-chunk peak exchange inside every step (the only collective; no
        # sample data crosses GPUs)
        self.sc = ShardedChain(self.cfg, local_rank, shard_frames_hint=self.n if world > 1 else 0, time_kernels=1,
                               fused=args.fused, subtrain_frames=args.subtrain, dc_overlap=args.dc_overlap)
        self.chain = self.sc.chain
        self.info = self.chain.info()
        self.replicas = False
        if world > 1:
            try:
                self.chain.seek(0)
            except gpu.IqGpuError:
                self.replicas = True   # FFT-filter / RMS-AGC chains are not exactly shardable (DESIGN.md 5): N independent replicas
        single = world == 1 or self.replicas
        self.single = single
        self.shard = self.sc.plan(self.n, 1)[0] if single else self.sc.plan(world * self.n, world)[rank]
        self.halo = self.shard.start - self.shard.lead
        self.raw = synth_torch(self.wl, self.shard.read_frames, dev, start=self.shard.lead)
        self.out = torch.empty(self.chain.out_capacity_frames(self.n + self.halo) * self.cfg.out_bytes, dtype=torch.uint8, device=dev)
        self.exchange = bool(self.sc.digital_agc and world > 1 and not self.replicas)
        self.produced = 0

    def step(self):
        st = self.stream.cuda_stream
        if self.single:
            self.chain.restart()
            self.produced = self.chain.process_device(self.raw.data_ptr(), self.n, self.out.data_ptr(), self.out.numel(), st)
        else:
            self.produced = self.sc.process_device(self.shard, self.raw.data_ptr(), self.out.data_ptr(), self.out.numel(), st,
                                                   None, self.dev)[0]
        return self.produced

    def timed(self, steps, warmup, sampler=None, min_seconds=0.0):
        """K steps (or, with min_seconds, as many whole batches of K as it takes) bracketed by CUDA events on the launch
        stream, barrier + synchronize on both sides, max over ranks.  Returns (ms total, steps run, t0, t1 wall)."""
        import torch.distributed as dist
        torch = self.torch
        for _ in range(warmup):
            self.step()
        self.chain.kernel_times(reset=True)
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        time.sleep(0.05)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0 = time.time()
        e0.record(self.stream)
        done = 0
        while True:
            for _ in range(steps):
                self.step()
            done += steps
            if min_seconds <= 0:
                break
            # the host runs far ahead of the device (no sync inside a batch): decide on the device's progress
            e1.record(self.stream)
            e1.synchronize()
            el = e0.elapsed_time(e1)
            if self.world > 1:          # every rank must take the same decision (the steps may hold a collective)
                t = torch.tensor([el], device=self.dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                el = float(t.item())
            if el >= 1e3 * min_seconds:
                break
        e1.record(self.stream)
        torch.cuda.synchronize()
        t1 = time.time()
        if self.world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, done, t0, t1

    def sharding_text(self):
        if self.world == 1:
            return "single stream"
        if self.replicas:
            return "replicas only (chain not exactly shardable)"
        if self.exchange:
            return "time shards; all-gather of per-chunk AGC peaks (4 B / 16384 frames), no sample data exchanged"
        return "time shards, no collective"


def run_file_bench(args):
    """--workload file:<cfg>: SURVEY 8(f) rank 2 — a raw capture on tmpfs through iqgpu_rawfile_run (reader thread -> chunk
    trains -> chain -> writer thread, pinned rings) into a raw file on tmpfs, timed by the wall clock like the reference's own
    run summary (src/main.c:286-306).  `value` and `e2e` are the same number here (the path is host to host by nature);
    cpu_baseline = the reference's stage code fed by read() / write() of the same file on a bounded prefix."""
    import numpy as np
    from iq_tool_b200 import baseline_workloads, gpu
    from iq_tool_b200.synth import synth_numpy
    name = args.workload.split(":", 1)[1]
    wl = baseline_workloads()[name]
    cfg = wl.config
    if gpu.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device; iq_tool_b200 has no CPU fallback")
    n = args.samples or (1 << 28)
    n -= n % 16384
    tmp = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    src, dst = os.path.join(tmp, f"iqgpu_bench_{os.getpid()}_in.raw"), os.path.join(tmp, f"iqgpu_bench_{os.getpid()}_out.raw")
    block = synth_numpy(wl, min(n, 1 << 24)).tobytes()
    nbytes = n * cfg.in_bytes
    with open(src, "wb") as f:
        left = nbytes
        while left:
            k = min(left, len(block))
            f.write(block[:k])
            left -= k
    steps = max(1, args.steps)
    try:
        sampler = ClockSampler(0)
        sampler.start()
        for _ in range(max(1, min(args.warmup, 2))):
            st = gpu.rawfile_run(cfg, src, dst, 0, args.train_chunks)
        t0 = time.time()
        p0 = time.perf_counter()
        for _ in range(steps):
            st = gpu.rawfile_run(cfg, src, dst, 0, args.train_chunks)
        dt = time.perf_counter() - p0
        clocks = sampler.stop(t0, time.time())
        out_bytes = os.path.getsize(dst)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, np.memmap(dst, dtype=np.uint8, mode="r").reshape(-1, cfg.out_bytes),
                         cfg.output_format)
        value = n * steps / dt / 1e6
        cpu = None
        if not args.no_cpu_baseline:
            from oracle.loader import CpuChain, have_ref
            kind = "ref_fast" if have_ref(fast=True) else "oracle"
            m = min(n, args.cpu_samples * 4)
            ch = CpuChain(cfg, kind)
            c0 = time.perf_counter()
            raw = np.fromfile(src, dtype=np.int16 if cfg.in_bytes == 4 else np.uint8, count=2 * m)
            out = ch.process(raw, threaded=(kind != "oracle"))
            out.tofile(dst + ".cpu")
            cdt = time.perf_counter() - c0
            os.remove(dst + ".cpu")
            cpu = {"value": m / cdt / 1e6, "unit": UNIT, "cores": 3 if kind != "oracle" else 1,
                   "kind": "reference" if kind != "oracle" else "port",
                   "sample": f"first {m} frames of the same file, read() -> reference stage code on the restated liquid layer "
                             f"(scalar dot products) -> write(); host has {os.cpu_count()} cpus"}
    finally:
        for pth in (src, dst):
            if os.path.exists(pth):
                os.remove(pth)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": steps, "warmup": args.warmup,
            "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": f"file:{wl.name}: raw file on {tmp} -> iqgpu_rawfile_run -> raw file; {wl.description}",
                       "frames_per_step": n, "output_frames_per_step": int(st.frames_out), "train_chunks": int(args.train_chunks or 64),
                       "trains_per_step": int(st.trains), "timing": "wall clock around the whole file run (open .. close)"},
            "roofline": None, "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": int(nbytes), "d2h_bytes_per_step": int(out_bytes),
                    "read_gbs": nbytes * steps / dt / 1e9},
            "gpu_launches": None, "clocks": clocks}
    print(json.dumps(line))
    return 0


DUMP_MAX_FRAMES = 1 << 21       # 2M frames: 16 MB of float32 I/Q (32 MB as float64) + 16 MB of float64 indices


def dump_outputs(path, frames, output_format, rank=0, world=1):
    """--dump-outputs: what the last timed step handed its caller, so two builds can be compared output for output.
    `frames` holds the output as rows of one frame's bytes (a CUDA tensor, a numpy array or a memory-mapped file).
    output.npy holds the frames as rows of float32 (float64 for 32-bit integer formats), output_index.npy their frame
    indices and frames_out.npy the frame count; both are stored as float64, which holds every count exactly.  Above
    DUMP_MAX_FRAMES a fixed, seeded sample of frames is stored.  With N > 1 every rank writes its own shard, with a
    _rank<r> suffix."""
    import numpy as np
    import torch
    from iq_tool_b200.configs import NUMPY_DTYPE
    nf = frames.shape[0]
    idx = np.arange(nf)
    if nf > DUMP_MAX_FRAMES:
        idx = np.sort(np.random.default_rng(20261020).choice(nf, DUMP_MAX_FRAMES, replace=False))
        frames = frames[torch.from_numpy(idx).to(frames.device)] if torch.is_tensor(frames) else frames[idx]
    raw = frames.cpu().numpy() if torch.is_tensor(frames) else np.asarray(frames)
    dt = np.dtype(NUMPY_DTYPE[output_format])
    vals = raw.view(dt).reshape(len(idx), -1)
    vals = vals.astype(np.float32 if dt.kind == "f" or dt.itemsize < 4 else np.float64)
    sfx = "" if world == 1 else f"_rank{rank}"
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, f"output{sfx}.npy"), vals)
    np.save(os.path.join(path, f"output_index{sfx}.npy"), idx.astype(np.float64))
    np.save(os.path.join(path, f"frames_out{sfx}.npy"), np.array([nf], dtype=np.float64))


def pcie_probe(world, dev, nbytes=1 << 30, reps=3):
    """Plain pinned-host -> device copies, all ranks at once: the platform's ceiling for the end-to-end leg, per rank.
    (SCALE_r01's box shows every GPU behind one NUMA node, `nvidia-smi topo`: CPU affinity 0-31, NUMA 0 — there is no
    placement to choose; this records what the host side of each GPU delivers when all of them pull together.)"""
    import torch
    import torch.distributed as dist
    host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    host.zero_()
    devb = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    devb.copy_(host, non_blocking=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        devb.copy_(host, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    gbs = reps * nbytes / (e0.elapsed_time(e1) / 1e3) / 1e9
    if world > 1:
        t = torch.zeros(world, device=dev, dtype=torch.float64)
        t[dist.get_rank()] = gbs
        dist.all_reduce(t)
        return [round(float(v), 2) for v in t.cpu().tolist()]
    return [round(gbs, 2)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--samples", type=int, default=0, help="input frames per GPU per step (default: workload's)")
    ap.add_argument("--cpu-samples", type=int, default=1 << 26,
                    help="input frames of the CPU sample: per step for --impl reference, x8 (about 10 s) for the cpu_baseline leg")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--fused", type=int, default=1)
    ap.add_argument("--dc-overlap", type=int, default=1)
    ap.add_argument("--subtrain", type=int, default=1 << 30, help="frames per sub-train (kernel launch group) of the HBM-resident leg")
    ap.add_argument("--e2e-subtrain", type=int, default=1 << 25, help="frames per sub-train of the host-buffer leg (H2D/compute/D2H pipeline depth)")
    ap.add_argument("--sustained-seconds", type=float, default=2.0, help="second timed leg: back-to-back steps for at least this long (0 = off)")
    ap.add_argument("--sharded-capture", default="cfg5",
                    help="second workload measured in the same run and reported as `sharded_capture` (BASELINE.json configs[4], the "
                         "multi-GPU configuration: time shards + the AGC peak all-gather); '' = off")
    ap.add_argument("--stage-leg", default="k1",
                    help="N = 1: a stage workload measured in the same run and reported as `stage_convert_shift` (k1: the "
                         "stand-alone convert + NCO shift pass, north_star's >= 60 %% of HBM target); '' = off")
    ap.add_argument("--no-pcie-probe", action="store_true")
    ap.add_argument("--train-chunks", type=int, default=64, help="file workloads: reference chunks per chain call")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the output of the last timed step to DIR/*.npy (a seeded sample when large)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    if args.workload.startswith("file:"):
        return run_file_bench(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    from iq_tool_b200 import gpu

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if gpu.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device; iq_tool_b200 has no CPU fallback")
    # one rank = one GPU = its own share of the host cores (the staging threads of the end-to-end leg stay put)
    try:
        cpus = sorted(os.sched_getaffinity(0))
        if world > 1 and len(cpus) >= 2 * world:
            per = len(cpus) // world
            os.sched_setaffinity(0, set(cpus[local_rank * per:(local_rank + 1) * per]))
    except (AttributeError, OSError):
        pass
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # an explicit (non-default) stream: the chain's kernels are launched on it and the timing events are recorded on it
    # (a NULL stream handle would make the chain use its own internal stream, invisible to torch's events)
    stream = torch.cuda.Stream(device=dev)
    stream.wait_stream(torch.cuda.current_stream())
    torch.cuda.set_stream(stream)

    run = WorkloadRun(args.workload, args, world, rank, local_rank, dev, stream, args.samples)
    wl, cfg, chain, n, halo = run.wl, run.cfg, run.chain, run.n, run.halo

    sampler = ClockSampler(local_rank)
    sampler.start()
    ms, steps_done, t0, t1 = run.timed(args.steps, args.warmup)
    clocks = sampler.stop(t0, t1)
    ktimes = chain.kernel_times(reset=True)
    launches_per_step = chain.info().kernel_launches
    produced = run.produced
    value = world * n * args.steps / (ms / 1e3) / 1e6
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, run.out[: produced * cfg.out_bytes].view(produced, cfg.out_bytes), cfg.output_format,
                     rank, world)

    # ---- sustained leg: the same step back to back for >= 2 s (power / clock behaviour of a long run) ----
    sustained = None
    if args.sustained_seconds > 0:
        s2 = ClockSampler(local_rank)
        s2.start()
        sms, sdone, st0, st1 = run.timed(args.steps, 1, min_seconds=args.sustained_seconds)
        sclk = s2.stop(st0, st1)
        chain.kernel_times(reset=True)
        sustained = {"value": world * n * sdone / (sms / 1e3) / 1e6, "unit": UNIT, "seconds": sms / 1e3, "steps": sdone,
                     "ms_per_step": sms / sdone, "clocks": sclk}

    # ---- end-to-end: host buffers through the C ABI (pinned host memory, H2D + D2H inside) ----
    e2e = None
    if args.e2e_steps > 0:
        import ctypes as C
        raw, out, shard, sc, exchange = run.raw, run.out, run.shard, run.sc, run.exchange
        nbytes = (n + halo) * cfg.in_bytes
        hin = gpu.lib.iqgpu_host_alloc(nbytes)
        hout = gpu.lib.iqgpu_host_alloc(out.numel())
        if hin and hout:
            torch.cuda.synchronize()
            # fill the pinned input from the device capture (outside the timed region)
            host_in = torch.frombuffer((C.c_uint8 * nbytes).from_address(hin), dtype=torch.uint8)
            host_in.copy_(raw.view(torch.uint8))
            nout = C.c_size_t(0)
            # the host-buffer leg pipelines H2D / compute / D2H over sub-trains: its own chain with shorter sub-trains
            e2e_chain = chain if exchange else gpu.Chain(cfg, local_rank, fused=args.fused, subtrain_frames=args.e2e_subtrain)
            host_out = torch.frombuffer((C.c_uint8 * out.numel()).from_address(hout), dtype=torch.uint8)
            def e2e_step():
                if exchange:
                    # sharded digital AGC: the peak exchange sits between the two halves of the device call
                    raw.view(torch.uint8).copy_(host_in, non_blocking=True)
                    k = sc.process_device(shard, raw.data_ptr(), out.data_ptr(), out.numel(), stream.cuda_stream, None, dev)[0]
                    host_out[: k * cfg.out_bytes].copy_(out[: k * cfg.out_bytes], non_blocking=True)
                    torch.cuda.synchronize()
                    nout.value = k
                    return
                if run.single:
                    e2e_chain.restart()
                else:
                    e2e_chain.seek(shard.lead)
                gpu._check(gpu.lib.iqgpu_chain_process(e2e_chain._h, hin, n + halo, None, 0, hout, out.numel(),
                                                       C.byref(nout), None))
            e2e_step()
            if world > 1:
                dist.barrier()
            tt0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                e2e_step()
            dt_own = time.perf_counter() - tt0
            dt = dt_own
            per_rank_s = [dt_own]
            if world > 1:
                t = torch.zeros(world, device=dev, dtype=torch.float64)
                t[rank] = dt_own
                dist.all_reduce(t)
                per_rank_s = [float(v) for v in t.cpu().tolist()]
                dt = max(per_rank_s)
            e2e = {"value": world * n * args.e2e_steps / dt / 1e6, "unit": UNIT,
                   "h2d_bytes_per_step": int(nbytes), "d2h_bytes_per_step": int(nout.value * cfg.out_bytes),
                   "steps": args.e2e_steps, "host_memory": "pinned (iqgpu_host_alloc)",
                   "per_rank_gbs_h2d": [round(nbytes * args.e2e_steps / s_ / 1e9, 2) for s_ in per_rank_s]}
            gpu.lib.iqgpu_host_free(hin)
            gpu.lib.iqgpu_host_free(hout)
            if not exchange:
                e2e_chain.close()
        if not args.no_pcie_probe:
            probe = pcie_probe(world, dev)
            if e2e is not None:
                # what plain pinned copies reach on the same box with every rank copying at once: the leg's ceiling
                e2e["pcie_probe_gbs_h2d_per_rank"] = probe
                e2e["fraction_of_probe_min_rank"] = round(min(e2e["per_rank_gbs_h2d"]) / max(min(probe), 1e-9), 3)

    # ---- BASELINE.json configs[4], the multi-GPU configuration, in the same run: cfg5 time-sharded with the peak exchange ----
    sharded = None
    if args.sharded_capture and args.sharded_capture != args.workload:
        del run.raw, run.out
        run2 = WorkloadRun(args.sharded_capture, args, world, rank, local_rank, dev, stream)
        k2 = max(5, min(args.steps, 20))
        ms2, _, _, _ = run2.timed(k2, 3)
        kt2 = run2.chain.kernel_times(reset=True)
        # where the exchange's time goes (a few extra steps with CUDA events around its three parts, per rank)
        exch = None
        if run2.exchange:
            run2.sc.exchange_marks = []
            for _ in range(5):
                run2.step()
            torch.cuda.synchronize()
            marks = [m for m in run2.sc.exchange_marks if len(m) == 4]
            run2.sc.exchange_marks = None
            if marks:
                mine_ms = [sum(m[i].elapsed_time(m[i + 1]) for m in marks) / len(marks) for i in range(3)]
                t = torch.zeros(world * 3, device=dev, dtype=torch.float64)
                t[3 * rank: 3 * rank + 3] = torch.tensor(mine_ms, dtype=torch.float64)
                dist.all_reduce(t)
                tt = t.cpu().tolist()
                exch = {"per_rank_ms": {"all_gather_incl_wait": [round(tt[3 * r], 4) for r in range(world)],
                                        "advance_over_lower_shards": [round(tt[3 * r + 1], 4) for r in range(world)],
                                        "own_scan_scale_convert": [round(tt[3 * r + 2], 4) for r in range(world)]}}
        sharded = {"workload": f"{run2.wl.name}: {run2.wl.description}", "value": world * run2.n * k2 / (ms2 / 1e3) / 1e6,
                   "unit": UNIT, "n_gpus": world, "steps": k2, "ms_per_step": ms2 / k2, "frames_per_gpu_per_step": run2.n,
                   "halo_frames": run2.halo, "sharding": run2.sharding_text(), "scaling": "weak",
                   "kernel_ms_per_step": {k: v[0] / k2 for k, v in kt2.items()}, "exchange": exch,
                   "note": "efficiency at N = value(N) / (N * value(1)) of THIS object across the per-N lines"}
        del run2

    # ---- north_star's other stage target in the driver's record: the stand-alone convert + NCO shift pass (k1) against HBM ----
    stage = None
    if args.stage_leg and world == 1 and args.stage_leg != args.workload:
        run3 = WorkloadRun(args.stage_leg, args, world, rank, local_rank, dev, stream)
        k3 = 10
        ms3, _, _, _ = run3.timed(k3, 3)
        kt3 = run3.chain.kernel_times(reset=True)
        bps3 = class_bytes_per_sample(run3.cfg, run3.chain.info())
        if kt3:
            # the stage north_star names is the convert + shift pass (class `pre`); k1's cf32 output pass is reported beside it
            d3 = "pre" if "pre" in kt3 else max(kt3.items(), key=lambda kv: kv[1][0])[0]
            per3 = kt3[d3][0] / max(1, kt3[d3][1])
            hbm3, src3, _ = load_peaks()
            ach3 = bps3.get(d3, 0.0) * run3.n * k3 / max(1, kt3[d3][1]) / (per3 / 1e3) / 1e9 if per3 > 0 else 0.0
            stage = {"workload": f"{run3.wl.name}: {run3.wl.description}", "value": run3.n * k3 / (ms3 / 1e3) / 1e6, "unit": UNIT,
                     "steps": k3, "ms_per_step": ms3 / k3, "frames_per_step": run3.n,
                     "roofline": {"bound": "hbm", "kernel": d3, "achieved": ach3, "peak": hbm3, "unit": "GB/s",
                                  "frac": ach3 / hbm3, "peak_source": src3, "launch_ms": per3,
                                  "algorithmic_bytes_per_input_frame": bps3.get(d3, 0.0)},
                     "kernel_ms_per_step": {k: v[0] / k3 for k, v in kt3.items()}}
        del run3

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel class ----
    hbm_peak, peak_src, peaks = load_peaks()
    bps = class_bytes_per_sample(cfg, chain.info())       # after the run: fused_front is known
    dom = max(ktimes.items(), key=lambda kv: kv[1][0])[0] if ktimes else None
    roofline = None
    if dom:
        dom_ms, dom_groups = ktimes[dom]
        per_launch_ms = dom_ms / max(1, dom_groups)
        frames_per_launch = (n + halo) * args.steps / max(1, dom_groups)
        alg_bytes = bps.get(dom, 0.0) * frames_per_launch
        achieved = alg_bytes / (per_launch_ms / 1e3) / 1e9 if per_launch_ms > 0 else 0.0
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                tj = json.load(f)
            if tj.get(dom, {}).get("bytes_per_input_frame") and tj[dom].get("workload", wl.name) == wl.name:
                traffic = tj[dom]["bytes_per_input_frame"] * frames_per_launch
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                    "launch_ms": per_launch_ms, "algorithmic_bytes_per_launch": alg_bytes,
                    "algorithmic_bytes_per_input_frame": bps.get(dom, 0.0),
                    "share_of_step": dom_ms / (ms if world == 1 else sum(v[0] for v in ktimes.values()))}
        if dom == "fused_front" and dc_local_state(cfg, chain.info()):
            roofline["note"] = ("launch_ms spans the front kernel, the DC stretch scan and the closed-form DC correction of the cf32 "
                                "tail; the correction of the resampled stream is added by the FIR behind the resampler while it "
                                "stages its tiles when there is one (cfg2), else by a read-modify-write pass that is inside "
                                "launch_ms and NOT counted as algorithmic traffic (SURVEY 8(d): input + 8 r)")
    flops = chain_flops_per_sample(cfg, run.info)
    fp32_peak_nominal = 148 * 128 * 2 * 1.965e9 / 1e12
    try:
        fp32_measured = gpu.fp32_peak_tflops(local_rank)
    except gpu.IqGpuError:
        fp32_measured = None
    ach = flops * value * 1e6 / world / 1e12
    fp32 = {"achieved_tflops": ach, "peak_tflops_measured": fp32_measured,
            "frac_of_measured": (ach / fp32_measured) if fp32_measured else None,
            "peak_source": "FFMA2 micro-benchmark in libiqgpu.so (iqgpu_ubench_fp32_peak), this run",
            "peak_tflops_nominal": fp32_peak_nominal, "frac_of_nominal": ach / fp32_peak_nominal,
            "flops_per_input_sample": flops}

    # ---- CPU baseline on a bounded sample (rank 0, N = 1 only) ----
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        from iq_tool_b200.synth import synth_torch
        from oracle.loader import CpuChain, have_ref
        kind = "ref_fast" if have_ref(fast=True) else "oracle"
        m = min(n, 8 * args.cpu_samples)          # about 10 s of CPU work at ~50 Msamples/s
        sample = synth_torch(wl, m, dev).cpu().numpy()
        ch = CpuChain(cfg, kind)
        ch.process(sample[: 2 * (1 << 20)], threaded=(kind != "oracle"))
        ch = CpuChain(cfg, kind)
        tt0 = time.perf_counter()
        ch.process(sample, threaded=(kind != "oracle"))
        dt = time.perf_counter() - tt0
        cpu = {"value": m / dt / 1e6, "unit": UNIT, "cores": 3 if kind != "oracle" else 1,
               "kind": "reference" if kind != "oracle" else "port",
               "sample": f"first {m} frames of the same capture; reference stage sources on the restated liquid "
                         f"layer (SCALAR dot products: a floor for a real AVX libliquid, not its speed), one thread per "
                         f"stage (pre/resampler/post) as pipeline.c:99-116; host has {os.cpu_count()} cpus"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{wl.name}: {wl.description}", "frames_per_gpu_per_step": n, "halo_frames": halo,
                   "output_frames_per_step": int(produced), "l2_policy": "inputs larger than L2 (no flush needed)",
                   "sharding": run.sharding_text(),
                   "fused_front": int(chain.info().fused_front),
                   "chunk_frames": 16384},
        "roofline": roofline, "fp32": fp32, "cpu_baseline": cpu, "e2e": e2e, "sustained": sustained,
        "sharded_capture": sharded, "stage_convert_shift": stage,
        "gpu_launches": int(launches_per_step) * args.steps, "clocks": clocks,
        "kernel_ms_per_step": {k: v[0] / args.steps for k, v in ktimes.items()},
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
