"""Several channels out of one capture: one iqgpu_chain_process_multi call against K iqgpu_chain_process calls, and one
iqgpu_rawfile_run_channels against K iqgpu_rawfile_run, for cfg5 (61.44 Msps -> 744187.5 sps, pre shift, digital AGC)
with K different shifts.

Host-buffer leg: a cs16 capture in pinned memory, outputs into pinned buffers; both forms end in a device synchronise
(the library's host path synchronises before it returns), the two forms alternate, each is repeated.  File leg: a raw
capture on tmpfs (page cache, no disk), the outputs on tmpfs too.  Prints one JSON line per measurement and writes them,
with the card's name and power limit read in the same run, to --out."""
from __future__ import annotations

import argparse
import ctypes as C
import dataclasses
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from iq_tool_b200 import baseline_workloads, gpu  # noqa: E402
from iq_tool_b200.synth import synth_numpy  # noqa: E402


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?", "?"])[:3]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def shifts(k: int) -> list[float]:
    # K stations spread over +-25 MHz of the 61.44 MHz capture
    return [float(-25e6 + 50e6 * (i + 0.5) / k) for i in range(k)]


def pinned(nbytes: int):
    p = gpu.lib.iqgpu_host_alloc(nbytes)
    if not p:
        raise RuntimeError("pinned allocation failed")
    return p, np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(p))


def host_leg(frames: int, ks: list[int], reps: int, emit) -> None:
    wl = baseline_workloads()["cfg5"]
    base = wl.config
    in_bytes = frames * base.in_bytes
    pin_in, view = pinned(in_bytes)
    block = synth_numpy(wl, 1 << 24).view(np.uint8)     # a seeded 64 MiB capture, repeated to fill the buffer
    for at in range(0, in_bytes, block.size):
        n = min(block.size, in_bytes - at)
        view[at:at + n] = block[:n]
    for k in ks:
        cfgs = [dataclasses.replace(base, freq_shift_hz=s) for s in shifts(k)]
        chains = [gpu.Chain(c, 0, subtrain_frames=1 << 25) for c in cfgs]
        cap = chains[0].out_capacity_frames(frames) * base.out_bytes
        outs = [pinned(cap) for _ in chains]
        handles = (C.c_void_p * k)(*[c._h for c in chains])
        out_ptrs = (C.c_void_p * k)(*[o[0] for o in outs])
        caps = (C.c_size_t * k)(*[cap] * k)
        nout = (C.c_size_t * k)()

        def multi():
            gpu._check(gpu.lib.iqgpu_chain_process_multi(handles, k, pin_in, frames, None, 0, out_ptrs, caps, nout, None))

        def separate():
            one = C.c_size_t()
            for i, ch in enumerate(chains):
                gpu._check(gpu.lib.iqgpu_chain_process(ch._h, pin_in, frames, None, 0, out_ptrs[i], cap, C.byref(one), None))

        for f in (multi, separate):          # warm-up: staging allocation, module load
            f()
        t = {"multi": [], "separate": []}
        for _ in range(reps):
            for name, f in (("multi", multi), ("separate", separate)):
                t0 = time.perf_counter()
                f()
                t[name].append(time.perf_counter() - t0)
        for name, ts in t.items():
            best, med = min(ts), float(np.median(ts))
            emit({"leg": "host_buffer", "form": name, "K": k, "frames": frames, "reps": reps,
                  "median_s": med, "min_s": best, "max_s": max(ts),
                  "h2d_bytes_per_call": in_bytes * (1 if name == "multi" else k),
                  "msamples_per_s_per_channel": frames / med / 1e6, "msamples_per_s_aggregate": k * frames / med / 1e6})
        for c in chains:
            c.close()
        for p, _ in outs:
            gpu.lib.iqgpu_host_free(p)
    gpu.lib.iqgpu_host_free(pin_in)


def file_leg(file_bytes: int, ks: list[int], reps: int, tmpdir: str, emit) -> None:
    wl = baseline_workloads()["cfg5"]
    base = wl.config
    frames = file_bytes // base.in_bytes
    d = tempfile.mkdtemp(prefix="iqchannels_", dir=tmpdir)
    try:
        src = os.path.join(d, "capture.cs16")
        block = synth_numpy(wl, 1 << 24).tobytes()      # 64 MiB, repeated
        with open(src, "wb") as f:
            left = frames * base.in_bytes
            while left:
                n = min(left, len(block))
                f.write(block[:n])
                left -= n
        for k in ks:
            cfgs = [dataclasses.replace(base, freq_shift_hz=s) for s in shifts(k)]
            outs = [os.path.join(d, f"out{i}.cs16") for i in range(k)]

            def multi():
                gpu.rawfile_run_channels(cfgs, src, outs)

            def separate():
                for c, o in zip(cfgs, outs):
                    gpu.rawfile_run(c, src, o)

            t = {"multi": [], "separate": []}
            for _ in range(reps):
                for name, f in (("multi", multi), ("separate", separate)):
                    t0 = time.perf_counter()
                    f()
                    t[name].append(time.perf_counter() - t0)
            for name, ts in t.items():
                med = float(np.median(ts))
                emit({"leg": "file", "form": name, "K": k, "frames": frames, "file_bytes": frames * base.in_bytes,
                      "reps": reps, "median_s": med, "min_s": min(ts), "max_s": max(ts),
                      "h2d_bytes_per_run": frames * base.in_bytes * (1 if name == "multi" else k),
                      "msamples_per_s_per_channel": frames / med / 1e6, "msamples_per_s_aggregate": k * frames / med / 1e6})
            for o in outs:
                os.remove(o)
    finally:
        shutil.rmtree(d, ignore_errors=True)


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--frames", type=int, default=1 << 28, help="host-buffer leg: capture frames (cs16)")
    ap.add_argument("--ks", default="1,2,4,8,16", help="host-buffer leg: channel counts")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--file-bytes", type=int, default=4 << 30, help="file leg: raw capture size (0 = skip the leg)")
    ap.add_argument("--file-ks", default="1,4,8")
    ap.add_argument("--file-reps", type=int, default=3)
    ap.add_argument("--tmpdir", default="/dev/shm", help="file leg: where the capture and outputs go (tmpfs)")
    ap.add_argument("--out", default="", help="also write the JSON lines here")
    a = ap.parse_args()
    if gpu.device_count() < 1:
        raise SystemExit("channels_timing: no CUDA device")
    lines = []

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)

    emit({"card": card()})
    host_leg(a.frames, [int(x) for x in a.ks.split(",")], a.reps, emit)
    if a.file_bytes:
        file_leg(a.file_bytes, [int(x) for x in a.file_ks.split(",")], a.file_reps, a.tmpdir, emit)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
