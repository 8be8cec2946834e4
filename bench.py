#!/usr/bin/env python
"""bench.py — Msamples/s of the Mode S decode hot path on B200 (see DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W            # this framework (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path, all host cores
    python bench.py --workload df17_aggressive|tiled_64g|snr_sweep ...   # BASELINE.json configs[2..4]
    python bench.py --workload receivers --receivers 256               # SURVEY 8(f) item 4: many receivers, one GPU
    python bench.py ... --dump-outputs DIR                              # also write what the last timed step computed to DIR/*.npy

Default workload (BASELINE.json configs[1]): a synthetic stand-in for testfiles/modes1.bin (its length,
seeded) tiled back to back to 1 GiB (536 870 912 samples = 4096 reference buffers) per GPU, --no-fix.
Weak scaling: rank r holds the r-th GiB of the tiled stream.  A step = one pass of the hot path over the rank's GiB:
  value : inputs resident in HBM; scan + frame-evaluation kernels, every rank on its own shard with
          its outputs in its own HBM (no data-path collective); CUDA events on the launching stream,
          max over ranks.
  e2e   : the same GiB from pinned HOST memory through the public API to decoded messages on the
          host: H2D, kernels, D2H of the records over the rank's own PCIe link, and the sequential
          half resolved by every rank for its own shard (sharded.resolve_distributed: only 4 KiB
          address caches travel between ranks); wall clock between barriers, max over ranks.
One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import ctypes
import hashlib
import json
import os
import queue
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
for p in (str(ROOT), str(ROOT / "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

GIB = 1 << 30
METRIC = "Msamples/s (2 MHz u8 IQ) decoded, whole job"

WORKLOADS = {
    # name: (description, decoder flags, bytes per GPU and step, device batches per step)
    "tiled_nofix": dict(desc="synthetic stand-in for modes1.bin tiled to 1 GiB per GPU, --no-fix (BASELINE.json configs[1])",
                        flags="--no-fix",
                        cfg=dict(fix_errors=0), nbytes=GIB, batches=1),
    "df17_aggressive": dict(desc="synthetic 2 MHz IQ with injected DF17 (0/1/2/3 flipped bits in turn), 1 GiB per GPU, "
                                 "full path with --aggressive two-bit repair (BASELINE.json configs[2])",
                            flags="--aggressive", cfg=dict(fix_errors=1, aggressive=1), nbytes=GIB, batches=1),
    "tiled_64g": dict(desc="synthetic stand-in for modes1.bin tiled to 8 GiB per GPU (64 GiB on 8 GPUs), --no-fix, buffer-per-GPU shards "
                           "(BASELINE.json configs[3])", flags="--no-fix", cfg=dict(fix_errors=0), nbytes=8 * GIB, batches=2),
}


def load_capture() -> tuple[np.ndarray, str]:
    """A synthetic stand-in for the reference's modes1.bin (same length, seeded): the input this
    benchmark has always used where the capture was not installed, generated, so it is the same
    wherever the benchmark runs and comparable with earlier builds' results."""
    from dump1090_b200 import synth
    return synth.random_traffic(356868, 560, seed=1), "synthetic stand-in for modes1.bin (356 868 samples, seed 1) tiled"


def df17_capture() -> tuple[np.ndarray, str]:
    """configs[2]: DF17 frames every 700 samples at 60 LSB over sigma = 1.5 noise, flipped bits cycling
    0, 1, 2, 3 (dump1090.c:854-894 repairs 1, with --aggressive 2, never 3): 16 MiB, then tiled."""
    from dump1090_b200 import synth
    return synth.df17_grid(8 << 20, 700, 5), "synthetic DF17 grid (period 700 samples, 0/1/2/3 flipped bits) tiled"


def shard_bytes(capture: np.ndarray, rank: int, nbytes: int = GIB) -> np.ndarray:
    """Bytes [rank*nbytes, (rank+1)*nbytes) of the capture tiled back to back."""
    start = (rank * nbytes) % capture.size
    reps = -(-(nbytes + start) // capture.size)
    return np.tile(capture, reps)[start: start + nbytes]


def workload_source(name: str):
    return df17_capture() if name == "df17_aggressive" else load_capture()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed regions run (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v == "Active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def base_config(name: str, world: int) -> dict:
    """The keys both arms report identically (the driver compares the two `config` dicts)."""
    w = WORKLOADS[name]
    return {"workload": w["desc"], "flags": w["flags"], "samples_per_gpu_step": w["nbytes"] // 2,
            "samples_per_step": world * (w["nbytes"] // 2),
            "l2_policy": "a step's input (>= 1 GiB per GPU) is larger than the 126 MB L2 (and than the host's last-level "
                         "cache for the CPU arm); no explicit flush"}


# ----------------------------------------------------------------------------- reference arm

def host_cpu_facts() -> dict:
    """What the CPU arm's number depends on besides the code: cores the process may use, the cgroup's
    CPU quota, SMT."""
    facts = {"affinity_cpus": len(os.sched_getaffinity(0)), "os_cpu_count": os.cpu_count()}
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        facts["cgroup_cpu_max"] = f"{quota} {period}"
        if quota != "max":
            facts["cgroup_cpus"] = round(int(quota) / int(period), 2)
    except Exception:
        facts["cgroup_cpu_max"] = None
    try:
        sib = Path("/sys/devices/system/cpu/cpu0/topology/thread_siblings_list").read_text().strip()
        facts["smt_siblings_cpu0"] = sib
        facts["threads_per_core"] = len(sib.replace("-", ",").split(","))
    except Exception:
        pass
    return facts


def effective_cores(facts: dict) -> int:
    n = facts["affinity_cpus"]
    if facts.get("cgroup_cpus"):
        n = min(n, max(1, int(facts["cgroup_cpus"])))
    return max(1, n)


_REF_DATA = None
_REF_FLAGS = (0, 0)


def _ref_worker(args):
    lo, hi = args
    import checker
    fix, aggressive = _REF_FLAGS
    t0 = time.perf_counter()
    fn = checker.ref_time if checker.REF_SO.exists() else checker.oracle_time
    fn(_REF_DATA[lo:hi], fix=fix, aggressive=aggressive, loops=1)
    return time.perf_counter() - t0


def run_reference(args) -> None:
    """The reference's own computeMagnitudeVector + detectModeS loop (oracle/_ref, compiled from the
    unmodified sources) on the host cores: one process per effective core on disjoint runs of whole
    buffers.  A step covers ONE GPU's share of the workload (1 GiB; the first GiB of an 8 GiB share):
    a bounded sample, the rate is what is compared."""
    global _REF_DATA, _REF_FLAGS
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    import checker
    name = args.workload
    if name == "receivers":
        print(json.dumps({"impl": "reference", "unavailable": "the reference serves one receiver per process: its rate per core is the tiled_nofix figure of this arm (147 Msamples/s = 73 receivers per core)"}))
        return
    if name == "snr_sweep":
        print(json.dumps({"impl": "reference", "unavailable": "snr_sweep compares detect rates; run --workload snr_sweep on the GPU arm, which times the oracle alongside"}))
        return
    kind = "reference" if checker.REF_SO.exists() else "port"
    if kind == "port":
        checker.build_oracle()
    w = WORKLOADS[name]
    capture, what = workload_source(name)
    facts = host_cpu_facts()
    cores = effective_cores(facts)
    sample_bytes = GIB
    _REF_DATA = shard_bytes(capture, 0, sample_bytes)
    _REF_FLAGS = (w["cfg"].get("fix_errors", 1), w["cfg"].get("aggressive", 0))
    nbuf = sample_bytes // 262144
    per = -(-nbuf // cores)
    slices = [(k * per * 262144, min(nbuf, (k + 1) * per) * 262144) for k in range(cores) if k * per < nbuf]
    ctx = mp.get_context("fork")
    worker_s = []
    with ctx.Pool(len(slices)) as pool:
        for _ in range(args.warmup):
            pool.map(_ref_worker, slices)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            worker_s += pool.map(_ref_worker, slices)
        dt = time.perf_counter() - t0
    value = args.steps * (sample_bytes // 2) / dt / 1e6
    per_worker = (sample_bytes // 2) / len(slices) / np.array(worker_s) / 1e6
    sample = (f"{what} to 1 GiB per step ({w['flags']}), {len(slices)} processes on disjoint buffer runs; "
              f"a step of this arm = one GPU's share of the workload, so its rate compares with the GPU arm's per GPU")
    cfg = base_config(name, args.gpus)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(value, 2), "unit": "Msamples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(1e3 * dt / args.steps, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic: " + what + " to 1 GiB per GPU",
        "config": cfg,
        "cpu_baseline": {"value": round(value, 2), "unit": "Msamples/s", "cores": len(slices), "kind": kind,
                         "sample": sample, "host": facts,
                         "per_worker_Msamples_s": {"min": round(float(per_worker.min()), 1),
                                                   "median": round(float(np.median(per_worker)), 1),
                                                   "max": round(float(per_worker.max()), 1)},
                         "worker_seconds": {"min": round(min(worker_s), 3), "median": round(float(np.median(worker_s)), 3),
                                            "max": round(max(worker_s), 3)}},
        "e2e": {"value": round(value, 2), "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ----------------------------------------------------------------------------- this framework

def so_digest() -> str:
    from dump1090_b200 import api
    return hashlib.sha256(Path(api.LIB_PATH).read_bytes()).hexdigest()[:16]


SCAN_KERNEL_SOURCES = ("dump1090_b200/csrc/modes_scan2.cu", "dump1090_b200/csrc/modes_scan_core.cuh",
                       "dump1090_b200/csrc/modes_internal.h")


def scan_source_digest() -> str:
    """sha256 over the files the scan kernel is compiled from and the compiler flags (the .so itself
    is not reproducible byte for byte: nvcc embeds per-build identifiers, so two builds of the same
    sources differ in their digests)."""
    h = hashlib.sha256()
    for rel in SCAN_KERNEL_SOURCES:
        h.update((ROOT / rel).read_bytes())
    for line in (ROOT / "Makefile").read_text().splitlines():
        if line.startswith(("ARCH", "NVFLAGS")):
            h.update(line.encode())
    return h.hexdigest()[:16]


def measured_traffic() -> tuple[float | None, str]:
    """DRAM bytes per scan-kernel launch from the committed ncu capture — only if it was taken with
    the scan kernel that is running now: profiles/scan_kernel_traffic.json records the digest of the
    kernel's sources + compiler flags (and the digest of the .so it was captured with)."""
    tp = ROOT / "profiles" / "scan_kernel_traffic.json"
    if not tp.exists():
        return None, "no capture committed"
    doc = json.loads(tp.read_text())
    if doc.get("so_sha256_16") == so_digest():
        return doc.get("dram_bytes_per_launch"), "profiles/scan_kernel_traffic.json (same library file)"
    if doc.get("scan_source_sha256_16") == scan_source_digest():
        return doc.get("dram_bytes_per_launch"), "profiles/scan_kernel_traffic.json (same scan-kernel sources and flags)"
    return None, (f"capture is of another scan kernel (sources {doc.get('scan_source_sha256_16')} != {scan_source_digest()}): "
                  "re-run scripts/ncu_traffic.sh")


def messages_digest(arr, n: int) -> str:
    """sha256 over (sample_pos, msgbits, msg) of the first n messages of a ctypes Message array."""
    h = hashlib.sha256()
    a = np.frombuffer(arr, dtype=np.uint8, count=n * 200).reshape(n, 200)
    h.update(np.ascontiguousarray(a[:, :14]).tobytes())                   # frame bytes
    h.update(np.ascontiguousarray(a[:, 16:24]).tobytes())                 # msgbits, msgtype
    h.update(np.ascontiguousarray(a[:, 192:200]).tobytes())               # sample_pos
    return h.hexdigest()


DUMP_SAMPLE = 65536           # rows of records / messages written by --dump-outputs (seeded choice when there are more)
MESSAGE_COLUMNS = ("sample_pos", "msgbits", "msgtype", "crcok", "crc", "errorbit", "phase_corrected")


def _sample_rows(n: int) -> np.ndarray:
    """A fixed, seeded choice of at most DUMP_SAMPLE row indices out of n, in increasing order."""
    if n <= DUMP_SAMPLE:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))


def dump_outputs(out_dir: Path, cands: np.ndarray, tiles: np.ndarray, messages, n_messages: int) -> None:
    """What the last timed step computed, as float64 arrays (every value is exact in float64):
      tile_counts.npy  records per scan tile of the last device batch (all tiles)
      records.npy      the batch's candidate records in tile order (the order is the stream's; the
                       array the kernels fill is in tile completion order), sampled: one row per
                       record = index, t, then per pass msg[14], msgtype, flags, errorbit, nfixed, crc
      messages.npy     the messages of the last end-to-end step, sampled: index, MESSAGE_COLUMNS, msg[14]
      counts.npy       [records, messages] before sampling"""
    out_dir.mkdir(parents=True, exist_ok=True)
    order = np.concatenate([np.arange(o, o + c) for o, c in tiles] or [np.zeros(0, np.int64)]).astype(np.int64)
    recs = cands[order]
    rows = _sample_rows(recs.size)
    r = recs[rows]
    p = r["p"]
    per_pass = [np.concatenate([p[:, k]["msg"], np.stack([p[:, k][f] for f in ("msgtype", "flags", "errorbit", "nfixed", "crc")], 1)], 1)
                for k in (0, 1)]
    np.save(out_dir / "tile_counts.npy", tiles["count"].astype(np.float64))
    np.save(out_dir / "records.npy", np.concatenate([rows[:, None], r["t"][:, None]] + per_pass, 1).astype(np.float64))
    m = np.ctypeslib.as_array(messages)[:n_messages]
    rows = _sample_rows(n_messages)
    m = m[rows]
    np.save(out_dir / "messages.npy", np.concatenate([rows[:, None], np.stack([m[f] for f in MESSAGE_COLUMNS], 1), m["msg"]], 1)
            .astype(np.float64))
    np.save(out_dir / "counts.npy", np.array([recs.size, n_messages], dtype=np.float64))


def run_ours(args) -> None:
    import torch
    import torch.distributed as dist
    from dump1090_b200 import api, sharded

    name = args.workload
    w = WORKLOADS[name]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # keep stdout clean for the one JSON line (NCCL prints its version banner there)
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the decode path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    host_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        host_group = dist.new_group(backend="gloo")        # 4 KiB address caches between the ranks' host threads
    dev = torch.device("cuda", local_rank)
    # Several ranks share this host's cores (and its cgroup CPU quota): each takes its share for the
    # threads that build message structs, and waits for its GPU asleep instead of spinning.
    host_share = None
    if world > 1:
        host_share = max(1, min(16, effective_cores(host_cpu_facts()) // world))
        os.environ.setdefault("MODES_BUILD_THREADS", str(host_share))
        if os.environ.get("BENCH_HOST_WAIT", "block") == "block":
            api.lib().modes_set_host_wait(1)
    numa = {"numa_node": None}
    if os.environ.get("BENCH_NUMA_BIND", "1") != "0":
        numa = sharded.bind_near_gpu(local_rank)              # before any pinned allocation
    trace = bool(os.environ.get("BENCH_E2E_TRACE"))
    if trace:
        print(f"rank {rank}: numa binding {numa}", file=sys.stderr)

    capture, what = workload_source(name)
    nbytes = w["nbytes"]
    nbuf = nbytes // api.BUFFER_BYTES
    nbatch = w["batches"]
    bbuf = nbuf // nbatch                                     # buffers per device batch (<= 4 GiB: positions are 32-bit)
    samples_per_gpu = nbytes // 2
    host_bytes = min(nbytes, GIB)                             # pinned host staging: 1 GiB, streamed repeatedly for larger shares
    pinned = api.PinnedBuffer(host_bytes)
    pinned.array[:] = shard_bytes(capture, rank, nbytes)[:host_bytes]
    carry0 = None
    if rank > 0:
        carry0 = bytes(shard_bytes(capture, rank - 1, nbytes)[-api.CARRY_BYTES:])
    d_iq = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    full = shard_bytes(capture, rank, nbytes) if nbytes > host_bytes else pinned.array
    for off in range(0, nbytes, GIB):
        d_iq[off: off + GIB].copy_(torch.from_numpy(np.ascontiguousarray(full[off: off + GIB])))
    carries = [carry0] + [bytes(full[b * bbuf * api.BUFFER_BYTES - api.CARRY_BYTES: b * bbuf * api.BUFFER_BYTES])
                          for b in range(1, nbatch)]
    del full

    cfg = dict(w["cfg"])
    dec = api.Decoder(device=local_rank, profile=1, **cfg)
    stream = torch.cuda.Stream(device=dev)
    dec.set_stream(stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def allmax(x: float) -> tuple[float, int]:
        """(max over ranks, rank that holds it)"""
        if world == 1:
            return x, 0
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        all_t = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(all_t, t)
        vals = [float(v.item()) for v in all_t]
        return max(vals), int(np.argmax(vals))

    def device_step():
        for b in range(nbatch):
            dec.detect_device(d_iq.data_ptr() + b * bbuf * api.BUFFER_BYTES, bbuf, carries[b])

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---- value: inputs resident in HBM, device-timed; nothing leaves the GPU, no rank waits for another
    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            device_step()
        barrier()
        dec.kernel_times_ms()                       # drop warm-up samples
        l0 = dec.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(args.steps):
            device_step()
        ev1.record(stream)
        barrier()
    dev_ms_rank = ev0.elapsed_time(ev1)
    launches = dec.launch_count() - l0
    ktimes = dec.kernel_times_ms()                  # per batch: scan, eval, both, batches
    n_cand = dec.detect_wait()
    last_records = dec.detect_fetch(bbuf) if args.dump_outputs and rank == 0 else None
    dev_ms, slow_rank = allmax(dev_ms_rank)
    scan_max, scan_rank = allmax(ktimes[0] * nbatch)
    eval_max, eval_rank = allmax(ktimes[1] * nbatch)
    value = world * samples_per_gpu * args.steps / (dev_ms * 1e-3) / 1e6

    # ---- H2D alone: one timed copy of the step's input over this rank's PCIe link
    h2d_ms = []
    host_t = torch.from_numpy(pinned.array)
    with torch.cuda.stream(stream):
        for k in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record(stream)
            for off in range(0, nbytes, host_bytes):
                d_iq[off: off + host_bytes].copy_(host_t, non_blocking=True)
            e1.record(stream)
            torch.cuda.synchronize(dev)
            h2d_ms.append(e0.elapsed_time(e1))
    h2d_only_ms, _ = allmax(min(h2d_ms))

    # ---- e2e: host buffers in, messages out, through the public API
    msg_cap = int(1.6 * 425744 * (nbytes // GIB)) + 4096 if name != "df17_aggressive" else (nbytes // 1400) * 2 + 4096
    parity = {"checked": False}
    if world == 1:
        dec2 = api.Decoder(device=local_rank, gpu_resolve=args.gpu_resolve, **cfg)
        out_arr = dec2.set_output_array(msg_cap)

        def e2e_step():
            dec2.reset()
            dec2.rearm_output()
            for off in range(0, nbytes, host_bytes):
                dec2.process_ptr(pinned.ptr, host_bytes)
            dec2.finish()
            return dec2.output_count()

        def e2e_join():
            return dec2.output_count()
    else:
        # Every rank: upload + kernels (records stay in its own HBM) -> records over its own PCIe
        # link -> its own host thread resolves its shard (resolve_distributed) while the main thread
        # uploads the next step.  No rank handles another rank's data.
        resolver = api.Resolver(**cfg)
        out_arr = resolver.set_output_array(msg_cap)
        xchg = sharded.ShmExchange(dist, host_group)     # the 4 KiB address caches travel through /dev/shm
        jobs, done = queue.Queue(), queue.Queue()
        rounds_seen, worker_ms, phase_ms = [], [], []
        pieces = nbytes // host_bytes                    # host staging is 1 GiB: larger shares go up piece by piece
        pbuf = host_bytes // api.BUFFER_BYTES
        rec_cap = (host_bytes // 2) // 64 + 4096
        land = [(api.PinnedBuffer(rec_cap * 56), api.PinnedBuffer(api.tiles_for(pbuf) * 8)) for _ in range(2)]
        slots = [None, None]                             # per pipeline slot: [(cands, tiles)] of the step's pieces

        def resolver_loop():
            while True:
                k = jobs.get()
                if k is None:
                    return
                try:
                    t0 = time.perf_counter()
                    parts = slots[k]
                    if len(parts) == 1:
                        cands, tiles = parts[0]
                    else:                                 # one shard = the pieces back to back
                        cands = np.concatenate([c for c, _ in parts])
                        tiles = np.concatenate([t for _, t in parts])
                        off_c = off_p = 0
                        nt = api.tiles_for(pbuf)
                        for i, (c, _) in enumerate(parts):
                            cands["t"][off_c: off_c + c.size] += (i * pbuf) << 17
                            tiles["offset"][off_p: off_p + nt] += off_c
                            off_c += c.size; off_p += nt
                    resolver.reset_state()
                    resolver.rearm_output()
                    info = sharded.resolve_distributed(resolver, cands, tiles, rank * nbuf, dist, host_group, exchange=xchg)
                    rounds_seen.append(info["rounds"])
                    phase_ms.append(info.get("ms") or {})
                    worker_ms.append(1e3 * (time.perf_counter() - t0))
                    done.put(None)
                except BaseException as e:               # surface it in e2e_join()
                    done.put(e)

        threading.Thread(target=resolver_loop, daemon=True).start()
        pending = [0]
        step_no = [0]

        def e2e_join():
            while pending[0]:
                err = done.get()
                pending[0] -= 1
                if err is not None:
                    raise err
            return resolver.output_count()

        # Pipeline (one 1 GiB piece per step): while batch i uploads and runs, batch i-1's records
        # come down the same link in the other direction (copy on a second stream out of a second
        # set of device buffers) and job i-1 — resolve + message structs — runs on the host thread.
        dbuf = [(torch.empty(rec_cap * 56, dtype=torch.uint8, device=dev),
                 torch.empty(api.tiles_for(pbuf) * 8, dtype=torch.uint8, device=dev)) for _ in range(2)]
        L = api.lib()
        in_flight = [None]                               # slot of the batch whose kernels are queued

        def fetch(k):
            n = dec.detect_wait()                        # the batch in slot k has finished
            cv = land[k][0].array.view(api.CANDIDATE_DTYPE)
            tv = land[k][1].array.view(api.TILE_DTYPE)
            return n, cv, tv

        def download(k, n, cv, tv):
            if n and L.modes_copy_to_host(api.C.c_void_p(cv.ctypes.data), api.C.c_void_p(dbuf[k][0].data_ptr()), n * 56):
                raise RuntimeError("record download failed")
            if L.modes_copy_to_host(api.C.c_void_p(tv.ctypes.data), api.C.c_void_p(dbuf[k][1].data_ptr()), tv.nbytes):
                raise RuntimeError("tile table download failed")
            return cv[:n], tv

        def hand_over(parts):
            e2e_join()                                   # the previous job is done on every rank (collective order)
            slots[0] = parts
            pending[0] += 1
            jobs.put(0)

        def e2e_step():
            if pieces > 1:                               # larger shares: piece by piece, no overlap of download and upload
                parts = []
                for i in range(pieces):
                    carry = carry0 if i == 0 else bytes(pinned.array[-api.CARRY_BYTES:])
                    dec.detect_host(pinned.ptr, pbuf, carry)
                    if i == 0:
                        e2e_join()
                    c, t = dec.detect_fetch_into(land[0][0].array.view(api.CANDIDATE_DTYPE), land[0][1].array.view(api.TILE_DTYPE))
                    parts.append((c.copy(), t.copy()))
                slots[0] = parts
                pending[0] += 1
                jobs.put(0)
                return 0
            k = step_no[0] & 1
            step_no[0] += 1
            prev = in_flight[0]
            got = fetch(prev) if prev is not None else None
            dec.detect_host(pinned.ptr, pbuf, carry0, dbuf[k][0].data_ptr(), rec_cap, dbuf[k][1].data_ptr())
            in_flight[0] = k
            if got is not None:
                hand_over([download(prev, *got)])
            return 0

        def e2e_flush():
            prev = in_flight[0]
            if prev is not None:
                got = fetch(prev)
                in_flight[0] = None
                hand_over([download(prev, *got)])

    def run_e2e(n_steps):
        with torch.cuda.stream(stream):
            barrier()
            t0 = time.perf_counter()
            for _ in range(n_steps):
                e2e_step()
            if world > 1:
                e2e_flush()
            n = e2e_join()
            barrier()
            return time.perf_counter() - t0, n

    _, e2e_msgs = run_e2e(min(args.warmup, 3))

    # ---- parity of the step just run (warm-up, outside the timed regions): the sequential resolver
    # over the same records, and the first 64 buffers against the CPU oracle
    try:
        import checker
        checker.build_oracle()
        n_mine = (dec2 if world == 1 else resolver).output_count()
        digest = messages_digest(out_arr, n_mine)
        dec.detect_device(d_iq.data_ptr(), bbuf, carry0)
        cands, tiles = dec.detect_fetch(bbuf)
        seq = api.Resolver(**cfg)
        seq_out = seq.set_output_array(msg_cap * (world if rank == 0 else 1))
        ok_seq = None
        if world == 1 and nbatch == 1:
            seq.run(cands, tiles, 0)
            ok_seq = messages_digest(seq_out, seq.output_count()) == digest and seq.output_count() == n_mine
        elif nbatch == 1:
            # all records to rank 0 once (gloo), resolved there sequentially, digests per shard compared
            blobs = [None] * world if rank == 0 else None
            dist.gather_object((cands.tobytes(), tiles.tobytes(), digest, n_mine), blobs, dst=0, group=host_group)
            if rank == 0:
                ok_seq = True
                for r, (cb, tb, dg, nm) in enumerate(blobs):
                    before = seq.output_count()
                    seq.run(np.frombuffer(cb, dtype=api.CANDIDATE_DTYPE), np.frombuffer(tb, dtype=api.TILE_DTYPE), r * nbuf)
                    part = (ctypes.c_uint8 * ((seq.output_count() - before) * 200)).from_buffer(seq_out, before * 200)
                    ok_seq &= (seq.output_count() - before == nm) and messages_digest(part, nm) == dg
        ok_oracle = None
        if rank == 0:
            k = 64
            head = np.ascontiguousarray(shard_bytes(capture, 0, nbytes)[: k * api.BUFFER_BYTES])
            exp, _ = checker.oracle_decode(head, fix=cfg.get("fix_errors", 1), aggressive=cfg.get("aggressive", 0), drop_eof=1,
                                           cap=400000)
            cut = k * api.BUFFER_SAMPLES - 240
            got = []
            for i in range(n_mine):
                if out_arr[i].sample_pos >= cut:
                    break
                got.append(out_arr[i].raw_line())
            ok_oracle = got == [m.hexline() for m in exp]
        parity = {"checked": True, "sequential_resolver_digest_equal": ok_seq, "first_64_buffers_equal_oracle": ok_oracle,
                  "messages_rank0": int(n_mine)}
    except Exception as e:                                    # the bench line still goes out; the failure is in it
        parity = {"checked": False, "error": repr(e)[:300]}

    e2e_steps = args.steps
    e2e_s_rank, e2e_msgs = run_e2e(e2e_steps)
    if last_records is not None:
        dump_outputs(Path(args.dump_outputs), *last_records, out_arr, (dec2 if world == 1 else resolver).output_count())
    e2e_s, e2e_slow = allmax(e2e_s_rank)
    if world > 1:
        t = torch.tensor([e2e_msgs], dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        e2e_msgs = int(t.item())
    e2e_value = world * samples_per_gpu * e2e_steps / e2e_s / 1e6
    d2h = n_cand * 56 * (nbytes // (bbuf * api.BUFFER_BYTES)) + api.tiles_for(nbuf) * 8 + 16

    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        peaks_path = ROOT / "MEASURED_PEAKS.json"
        if peaks_path.exists():
            peak, peak_src = float(json.loads(peaks_path.read_text())["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured)"
        else:
            peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        scan_ms = ktimes[0]                                   # per launch (= per device batch) on rank 0
        alg_bytes = 2 * (bbuf * api.BUFFER_SAMPLES)
        achieved = alg_bytes / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else 0.0
        traffic, traffic_src = measured_traffic()
        if traffic is not None and nbatch > 1:
            traffic, traffic_src = None, "capture is of the 1 GiB launch"

        cpu_baseline = None
        if world == 1 and name != "tiled_64g":
            import checker
            kind = "reference" if checker.REF_SO.exists() else "port"
            if kind == "port":
                checker.build_oracle()
            sample = pinned.array[: 512 << 20]
            fn = checker.ref_time if kind == "reference" else checker.oracle_time
            loops = 3 if name == "tiled_nofix" else 1
            secs = fn(sample, fix=cfg.get("fix_errors", 1), aggressive=cfg.get("aggressive", 0), loops=loops)
            cpu_baseline = {"value": round(loops * (sample.size // 2) / secs / 1e6, 2), "unit": "Msamples/s", "cores": 1,
                            "kind": kind,
                            "sample": f"first 512 MiB of the workload x {loops} loops, single thread (the reference's "
                                      f"own design: one decode thread), {w['flags']}"}
            if kind == "reference" and name == "tiled_nofix":
                try:                                    # the two hot calls separately (SURVEY.md 8(d)); never fatal
                    part = sample[: 256 << 20]
                    t_mag, t_det = checker.ref_time_phases(part, fix=0, loops=1)
                    n = part.size // 2
                    cpu_baseline["phases"] = {"computeMagnitudeVector_Msamples_s": round(n / t_mag / 1e6, 1),
                                              "detectModeS_Msamples_s": round(n / t_det / 1e6, 1),
                                              "sample": "first 256 MiB, one pass"}
                except Exception as e:
                    cpu_baseline["phases"] = {"error": repr(e)}

        conf = base_config(name, world)                      # the same dict in both arms
        step_facts = {"candidates_per_gpu_batch": n_cand, "device_batches_per_step": nbatch,
                      "step": "scan kernel (magnitude+preamble) + frame-evaluation kernel per device batch; every rank on its "
                              "own shard, outputs in its own HBM, no data-path collective"}
        out = {
            "metric": METRIC, "value": round(value, 1), "unit": "Msamples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dev_ms / args.steps, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic: " + what + f" to {nbytes // GIB} GiB per GPU",
            "config": conf, "step_facts": step_facts,
            "clocks": clocks, "gpu_launches": int(launches),
            "parity_checked": bool(parity.get("checked") and parity.get("first_64_buffers_equal_oracle")
                                   and parity.get("sequential_resolver_digest_equal") is not False),
            "parity": parity,
            "per_rank": {"step_ms_max": round(dev_ms / args.steps, 4), "slowest_rank": slow_rank,
                         "scan_ms_max": round(scan_max, 4), "scan_ms_max_rank": scan_rank,
                         "eval_ms_max": round(eval_max, 4), "eval_ms_max_rank": eval_rank,
                         "limiter": "kernels only: ranks are independent in the timed region"},
            "e2e": {"value": round(e2e_value, 1), "unit": "Msamples/s", "h2d_bytes_per_step": nbytes + 480 * nbatch,
                    "d2h_bytes_per_step": int(d2h), "messages_per_step": int(e2e_msgs),
                    "ms_per_step": round(1e3 * e2e_s / e2e_steps, 3), "slowest_rank": e2e_slow,
                    "h2d_only_ms": round(h2d_only_ms, 3),
                    "h2d_fraction_of_step": round(h2d_only_ms / (1e3 * e2e_s / e2e_steps), 3),
                    "path": ("modes_process()+modes_finish() from pinned host memory"
                             + (", order-dependent half on the device (gpu_resolve)" if args.gpu_resolve else "")) if world == 1 else
                            "per rank: modes_detect_host (H2D + kernels) + modes_detect_fetch (D2H of its records) + "
                            "resolve_distributed on its own host thread (4 KiB address caches through /dev/shm only); the "
                            "download of step i-1 and its resolve overlap the upload of step i"},
            "roofline": {"bound": "hbm", "kernel": "scan_kernel (fused magnitude + preamble tests)",
                         "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                         "scan_ms": round(scan_ms, 4), "eval_ms": round(ktimes[1], 4),
                         "batches_timed": int(ktimes[3]), "library_sha256_16": so_digest(),
                         "scan_source_sha256_16": scan_source_digest()},
            "cpu_baseline": cpu_baseline,
        }
        if world > 1:
            out["e2e"]["host_threads_per_rank"] = int(os.environ.get("MODES_BUILD_THREADS", "0")) or None
            out["e2e"]["host_wait"] = os.environ.get("BENCH_HOST_WAIT", "block")
            out["e2e"]["resolve_rounds_max"] = int(max(rounds_seen)) if rounds_seen else None
            out["e2e"]["resolve_worker_ms_median_rank0"] = round(float(np.median(worker_ms)), 2) if worker_ms else None
            try:                                        # where the worker's time goes; "exchange" includes waiting for the slowest rank
                keys = sorted({k for d in phase_ms for k in d})
                out["e2e"]["resolve_worker_phases_ms_median_rank0"] = {
                    k: round(float(np.median([d.get(k, 0.0) for d in phase_ms])), 2) for k in keys} if phase_ms else None
            except Exception as e:
                out["e2e"]["resolve_worker_phases_ms_median_rank0"] = {"error": repr(e)}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(out), flush=True)
        os.dup2(2, 1)
    if world > 1:
        jobs.put(None)
        dist.barrier()
        xchg.close()
        dist.destroy_process_group()


# ----------------------------------------------------------------------------- configs[4]: SNR sweep

def run_snr_sweep(args) -> None:
    """BASELINE.json configs[4]: injected DF17 preambles at low SNR, --aggressive, >= 10^4 frames per
    point split across the ranks; detect rate and messages/s on the GPUs, and the CPU oracle on the
    same streams — identical decisions required, not merely a similar rate.  SNR = pulse power /
    noise power in the 2 MHz sample stream = A^2 / (2 sigma^2).  The reference's demodulator (strict
    ordering of the 10 preamble samples, mean half-bit difference >= 2550/360 LSB, dump1090.c:1602-1726)
    decodes nothing below about +8 dB by this definition, so the points of BASELINE.json (-3..+6 dB)
    are followed by +8..+20 dB, where the detect rate climbs from 0 to 1."""
    import importlib.util
    import torch
    import torch.distributed as dist
    import checker
    from dump1090_b200 import api
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    spec = importlib.util.spec_from_file_location("snr_sweep", ROOT / "scripts" / "snr_sweep.py")
    sweep = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sweep)
    checker.build_oracle()
    frames_total = max(10000, args.frames)
    per_rank = -(-frames_total // world)
    dec = api.Decoder(device=local_rank, aggressive=1)
    points = []
    t_gpu_total = 0.0
    samples_total = 0
    for snr in list(range(-3, 7)) + [8, 10, 12, 14, 16, 18, 20]:
        data, truth = sweep.stream_at(float(snr), per_rank, 100000 + 1000 * snr + rank)
        dec.decode(data[: 262144 * 2])                        # warm
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        got = dec.decode(data)
        t_gpu = time.perf_counter() - t0
        t1 = time.perf_counter()
        exp, st = checker.oracle_decode(data, aggressive=1, cap=4 * per_rank + 4096)
        t_cpu = time.perf_counter() - t1
        same = [m.raw_line() for m in got] == [m.hexline() for m in exp] and list(dec.stats().values()) == st
        found = len({m.hex() for m in got} & truth)
        row = torch.tensor([per_rank, len(got), found, int(same), data.size // 2, t_gpu * 1e6, t_cpu * 1e6,
                            sum(1 for m in got if m.nfixed == 1), sum(1 for m in got if m.nfixed == 2)],
                           dtype=torch.float64, device=dev)
        if world > 1:
            rows = [torch.zeros_like(row) for _ in range(world)]
            dist.all_gather(rows, row)
        else:
            rows = [row]
        r = np.array([x.cpu().numpy() for x in rows])
        frames = int(r[:, 0].sum())
        t_g = float(r[:, 5].max()) * 1e-6
        points.append({"snr_db": snr, "frames": frames, "messages": int(r[:, 1].sum()),
                       "true_frames_recovered": int(r[:, 2].sum()), "detect_rate": round(float(r[:, 2].sum()) / frames, 4),
                       "gpu_equals_oracle": bool(r[:, 3].min() == 1), "fixed_1bit": int(r[:, 7].sum()), "fixed_2bit": int(r[:, 8].sum()),
                       "gpu_msgs_per_s": round(float(r[:, 1].sum()) / t_g, 1), "gpu_Msamples_s": round(float(r[:, 4].sum()) / t_g / 1e6, 1),
                       "oracle_Msamples_s_per_core": round(float(r[:, 4].sum()) / float(r[:, 6].sum()), 1)})
        t_gpu_total += t_g
        samples_total += int(r[:, 4].sum())
    if rank == 0:
        os.dup2(saved_stdout, 1)
        print(json.dumps({
            "metric": METRIC, "value": round(samples_total / t_gpu_total / 1e6, 1), "unit": "Msamples/s", "n_gpus": world,
            "steps": len(points), "warmup": 1, "ms_per_step": round(1e3 * t_gpu_total / len(points), 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic: injected DF17 over Gaussian noise",
            "config": {"workload": "low-SNR sweep: injected DF17 preambles, --aggressive, >= 10^4 frames per point across the "
                                   "ranks, host memory in, messages out (BASELINE.json configs[4])",
                       "flags": "--aggressive", "snr_definition": "A^2 / (2 sigma^2) in the 2 MHz sample stream; A = 20 LSB",
                       "frames_per_point": int(points[0]["frames"])},
            "parity_checked": all(p["gpu_equals_oracle"] for p in points), "points": points,
            "note": "value = end-to-end decode() of small streams (a few MB per point and rank): launch- and copy-latency "
                    "bound, not a throughput figure; the result of this workload is the detect-rate table and its equality "
                    "with the CPU oracle"}), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ----------------------------------------------------------------------------- SURVEY 8(f) item 4: many receivers

def run_receivers(args) -> None:
    """Many independent 2 MHz receivers on one GPU (modes_pool_*): every step takes ONE 131072-sample
    buffer from each of R receivers (pinned host memory in, messages out, per-receiver address caches and
    carries), i.e. the live-ingest shape of rtlsdrCallback (dump1090.c:442-456) batched across receivers
    instead of across time.  Receiver r's stream is the tiled capture starting r buffers in; receiver 0's
    messages are checked against the CPU oracle's decode of its stream."""
    import ctypes
    import torch
    import checker
    from dump1090_b200 import api
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(0)
    n_rx = max(1, args.receivers)
    steps, warm = max(1, args.steps), max(1, args.warmup)
    capture, what = load_capture()
    BUF = api.BUFFER_BYTES
    total = steps + warm
    # one pinned block: the tiled capture, long enough that receiver r can read buffers r .. r+total
    pinned = api.PinnedBuffer((n_rx + total) * BUF)
    pinned.array[:] = shard_bytes(capture, 0, (n_rx + total) * BUF)
    ids = np.arange(n_rx, dtype=np.uint32)
    first = []
    msgs = 0
    sampler = ClockSampler(0)
    with api.ReceiverPool(n_rx, fix_errors=0) as pool:
        # messages of all receivers land in one array (modes_pool_set_output), receiver 0's are kept for the check
        out, out_rx = pool.set_output_array(n_rx * 400 + 4096)

        msg_size = ctypes.sizeof(api.Message)
        raw0 = []                                       # receiver 0's messages as bytes, formatted after the timed region
        live = {}

        def submit(k):
            live[k] = (ctypes.c_void_p * n_rx)(*[pinned.ptr + (r + k) * BUF for r in range(n_rx)])
            pool.submit_ptrs(ids, live[k])

        def collect(k):
            pool.rearm_output()
            pool.collect(None)
            del live[k]
            n = pool.output_count()
            assert n <= len(out), "message array too small"
            m0 = int(np.searchsorted(out_rx[:n], 1))    # receivers are served in the order listed: receiver 0 first
            raw0.append(ctypes.string_at(out, m0 * msg_size))
            return n

        # two batches in flight: batch k+1 is uploaded and scanned while batch k is resolved on the host
        submit(0)
        for k in range(1, warm + 1):
            submit(k)
            collect(k - 1)
        torch.cuda.synchronize()
        sampler.start()
        t0 = time.perf_counter()
        for k in range(warm + 1, total + 1):
            if k < total:
                submit(k)
            msgs += collect(k - 1)
        dt = time.perf_counter() - t0
        clocks = sampler.stop()
        for blob in raw0:
            arr = (api.Message * (len(blob) // msg_size)).from_buffer_copy(blob)
            first.extend(m.raw_line() for m in arr)
        stats0 = list(pool.stats(0).values())
    exp, exp_stats = checker.oracle_decode(pinned.array[: total * BUF], fix=0, drop_eof=1, cap=4_000_000)
    ok = first == [m.hexline() for m in exp] and stats0 == exp_stats
    samples = n_rx * steps * 131072
    os.dup2(saved_stdout, 1)
    print(json.dumps({
        "metric": METRIC, "value": round(samples / dt / 1e6, 1), "unit": "Msamples/s", "n_gpus": 1, "steps": steps, "warmup": warm,
        "ms_per_step": round(1e3 * dt / steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": f"synthetic: {what}, receiver r starts r buffers in",
        "config": {"workload": f"{n_rx} independent receivers, one 131072-sample buffer of each per step through modes_pool_ingest "
                               "(SURVEY.md 8(f) item 4), --no-fix", "flags": "--no-fix", "receivers": n_rx,
                   "samples_per_step": n_rx * 131072, "h2d_bytes_per_step": n_rx * (BUF + api.CARRY_BYTES),
                   "device_bytes_scanned_per_step": 2 * n_rx * BUF,
                   "step": "modes_pool_submit(k+1) then modes_pool_collect(k): carries + buffers H2D, scan + frame evaluation over 2R "
                           "buffers (pad, data pairs) of one batch while the batch before it is fetched (records D2H) and resolved "
                           "per receiver on the host into one message array; wall clock"},
        "clocks": clocks, "messages_per_step": round(msgs / steps, 1),
        "receivers_in_real_time": int(samples / dt / 2e6),
        "parity_checked": bool(ok), "parity": {"receiver_0_equals_oracle_decode_of_its_stream": bool(ok), "messages_receiver_0": len(first)},
        "note": "value is end to end (host buffers in, messages out); one receiver delivers 2 M samples/s"}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 30; snr_sweep has its fixed set of points)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="tiled_nofix", choices=list(WORKLOADS) + ["snr_sweep", "receivers"])
    ap.add_argument("--receivers", type=int, default=256, help="receivers: independent streams, one buffer of each per step")
    ap.add_argument("--frames", type=int, default=10000, help="snr_sweep: frames per SNR point (whole job)")
    ap.add_argument("--gpu-resolve", type=int, default=0, help="N=1 e2e: 1 = the order-dependent half on the GPU too (modes_config.gpu_resolve)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0: candidate records, messages) to DIR/*.npy; "
                         "the decode workloads only (" + ", ".join(WORKLOADS) + "), not snr_sweep or receivers")
    args = ap.parse_args()
    if args.workload == "snr_sweep" and args.steps is not None:
        ap.error("snr_sweep times one decode at each of its 17 SNR points: --steps does not apply")
    if args.steps is None:
        args.steps = 30
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in WORKLOADS):
        ap.error(f"--dump-outputs needs the GPU decode workloads ({', '.join(WORKLOADS)})")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "snr_sweep":
        run_snr_sweep(args)
    elif args.workload == "receivers":
        run_receivers(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
