#!/usr/bin/env python
"""pool_resolve_bench.py — the receiver pool (modes_pool_*) with the order-dependent half on the host
(gpu_resolve = 0: one modes_resolver per receiver on MODES_POOL_THREADS threads, default 4) and on the
device (gpu_resolve = 1: one warp per receiver, address caches resident in HBM), alternating in one call.

    python scripts/pool_resolve_bench.py [--receivers 64,256,1024] [--steps 40] [--rounds 3] [--out FILE]

The workload is bench.py --workload receivers: receiver r reads the tiled synthetic stand-in for
modes1.bin r buffers in, --no-fix, one 131072-sample buffer of every receiver per step from one pinned
block, submit(k+1) / collect(k), all messages into one output array.  Per receiver count and mode:
  ms_per_step         wall clock over `steps` steps (each round ends with a collect, which waits for
                      the device), median of the rounds; the two modes run in turn, round by round
  cpu_s_per_step      user + system CPU seconds of the whole process (getrusage) over the same steps
  msgs_per_step
  d2h_bytes_per_step  device-to-host copies in the CUDA trace of a separate torch.profiler run
  kernel_us_per_step  the same run: pool_resolve_kernel (count + emit passes) + resolve_offsets_kernel
Checks: every warm-up step's output array and receiver_of are byte-identical between the modes, and
receiver 0's messages over all steps equal the CPU oracle's decode of its stream.  One JSON line per
receiver count and mode after a line naming the card and its power limit.
"""
from __future__ import annotations

import argparse
import ctypes
import hashlib
import json
import os
import resource
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

BUF = 262144


def card() -> dict:
    import torch
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def cpu_seconds() -> float:
    r = resource.getrusage(resource.RUSAGE_SELF)
    return r.ru_utime + r.ru_stime


class Run:
    """One pool and the steps it has taken: step k hands every receiver r buffer r + k of the block."""

    def __init__(self, api, pinned, n_rx: int, gpu_resolve: int):
        self.api, self.pinned, self.n = api, pinned, n_rx
        self.pool = api.ReceiverPool(n_rx, fix_errors=0, gpu_resolve=gpu_resolve)
        self.out, self.out_rx = self.pool.set_output_array(n_rx * 400 + 4096)
        self.ids = np.arange(n_rx, dtype=np.uint32)
        self.size = ctypes.sizeof(api.Message)
        self.k = 0
        self.live = {}
        self.raw0 = []                                   # receiver 0's messages, as bytes

    def _submit(self, k):
        self.live[k] = (ctypes.c_void_p * self.n)(*[self.pinned.ptr + (r + k) * BUF for r in range(self.n)])
        self.pool.submit_ptrs(self.ids, self.live[k])

    def _collect(self, k, digests):
        self.pool.rearm_output()
        self.pool.collect(None)
        del self.live[k]
        n = self.pool.output_count()
        assert n <= len(self.out), "message array too small"
        m0 = int(np.searchsorted(self.out_rx[:n], 1))   # receivers are served in the order listed: receiver 0 first
        self.raw0.append(ctypes.string_at(self.out, m0 * self.size))
        if digests is not None:
            digests.append(hashlib.sha256(ctypes.string_at(self.out, n * self.size) + self.out_rx[:n].tobytes()).hexdigest())
        return n

    def steps(self, count, digests=None) -> int:
        """`count` steps, two batches in flight, drained at the end; returns the messages."""
        k0, msgs = self.k, 0
        self._submit(k0)
        for k in range(k0 + 1, k0 + count):
            self._submit(k)
            msgs += self._collect(k - 1, digests)
        msgs += self._collect(k0 + count - 1, digests)
        self.k += count
        return msgs

    def receiver0(self) -> list:
        blob = b"".join(self.raw0)
        arr = (self.api.Message * (len(blob) // self.size)).from_buffer_copy(blob)
        return [m.raw_line() for m in arr]

    def close(self):
        self.pool.close()


def trace_totals(api, pinned, n_rx: int, gpu_resolve: int, steps: int) -> dict:
    """D2H bytes and the pool kernels' time per step from a torch.profiler run of its own."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    run = Run(api, pinned, n_rx, gpu_resolve)
    run.steps(2)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        run.steps(steps)
        torch.cuda.synchronize()
    run.close()
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    d2h = sum(int(e.get("args", {}).get("bytes", 0)) for e in events
              if e.get("cat") == "gpu_memcpy" and "DtoH" in e.get("name", ""))
    kernels = {}
    for e in events:
        if e.get("cat") == "kernel" and ("pool_resolve_kernel" in e["name"] or "resolve_offsets_kernel" in e["name"]):
            key = "pool_resolve_kernel<emit>" if "ILb1E" in e["name"] or "<true>" in e["name"] else \
                  "pool_resolve_kernel<count>" if "pool_resolve" in e["name"] else "resolve_offsets_kernel"
            kernels[key] = kernels.get(key, 0.0) + float(e["dur"])
    return {"d2h_bytes_per_step": round(d2h / steps), "kernel_us_per_step": {k: round(v / steps, 1) for k, v in sorted(kernels.items())},
            "trace_steps": steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--receivers", default="64,256,1024")
    ap.add_argument("--steps", type=int, default=40, help="timed steps per round and mode")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=6, help="untimed steps per mode, compared byte for byte")
    ap.add_argument("--trace-steps", type=int, default=8)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    import bench
    import checker
    from dump1090_b200 import api
    assert api.BUFFER_BYTES == BUF
    torch.cuda.set_device(0)
    lines = [dict(card(), script="scripts/pool_resolve_bench.py", steps=args.steps, rounds=args.rounds, warmup=args.warmup,
                  pool_threads=int(os.environ.get("MODES_POOL_THREADS", "4")), host_cpus=os.cpu_count())]
    print(json.dumps(lines[0]), flush=True)
    capture, what = bench.load_capture()
    for n_rx in [int(x) for x in args.receivers.split(",")]:
        total = args.warmup + args.rounds * args.steps
        pinned = api.PinnedBuffer((n_rx + total + args.trace_steps + 2) * BUF)
        pinned.array[:] = bench.shard_bytes(capture, 0, pinned.array.size)
        runs = [Run(api, pinned, n_rx, g) for g in (0, 1)]
        digests = [[], []]
        for g in (0, 1):
            runs[g].steps(args.warmup, digests[g])
        torch.cuda.synchronize()
        ms, cpu, msgs = [[], []], [[], []], [0, 0]
        for _ in range(args.rounds):
            for g in (0, 1):
                c0, t0 = cpu_seconds(), time.perf_counter()
                msgs[g] += runs[g].steps(args.steps)
                dt, dc = time.perf_counter() - t0, cpu_seconds() - c0
                ms[g].append(1e3 * dt / args.steps)
                cpu[g].append(dc / args.steps)
        exp, _ = checker.oracle_decode(pinned.array[: total * BUF], fix=0, drop_eof=1, cap=4_000_000)
        want0 = [m.hexline() for m in exp]
        same = digests[0] == digests[1]
        for g in (0, 1):
            got0 = runs[g].receiver0()
            runs[g].close()
            line = {"receivers": n_rx, "gpu_resolve": g, "ms_per_step": round(float(np.median(ms[g])), 3),
                    "ms_per_step_rounds": [round(x, 3) for x in ms[g]],
                    "cpu_s_per_step": round(float(np.median(cpu[g])), 5),
                    "msgs_per_step": round(msgs[g] / (args.rounds * args.steps), 1),
                    "receivers_in_real_time": int(n_rx * 131072 / (np.median(ms[g]) * 1e-3) / 2e6),
                    "warmup_outputs_identical_across_modes": same, "receiver_0_equals_oracle": got0 == want0,
                    "messages_receiver_0": len(got0), "data": f"synthetic: {what}, receiver r starts r buffers in, --no-fix"}
            line.update(trace_totals(api, pinned, n_rx, g, args.trace_steps))
            lines.append(line)
            print(json.dumps(line), flush=True)
        del runs, pinned
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
