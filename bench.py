#!/usr/bin/env python
"""bench.py -- input GB/s matched by the PFAC scan (BASELINE.json metric) on N B200s.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...                      (CPU port of the reference's scan, rank 0 only)
    python bench.py --workload config1|dictionary|config2|config3|config4 [--scaling strong] [--bytes B]
    python bench.py ... --dump-outputs DIR                    (the records of the last timed step as DIR/*.npy)

A "step" is one pass of the hot path over one rank's shard of the input:
  * `value`  : device-resident -- input already in HBM, one pfac_scan_device launch sequence per step,
               timed with CUDA events on the launching stream, max over ranks;
  * `e2e`    : the same shard through pfac_scan_host (pinned host buffer -> H2D -> kernels -> D2H of
               the compact records), host<->device copies inside the timed region.
Workload at N=1 = BASELINE.json configs[2] (the config the metric is quoted on): 10,000 synthetic
Snort-like patterns over 1 GiB of HTTP-like text, 4 streams per GPU.  For N>1 every rank scans its
own 1 GiB shard (+ halo from the next shard): weak scaling, no data-path collective; with
`--scaling strong` the workload's bytes are ONE input cut over the ranks by pfac_job_plan.
The K timed steps of `value` run with nothing between the kernels of a step; the dominant kernel's own duration
(`roofline`) comes from K more steps with a CUDA-event pair around that kernel.  Shards smaller than the L2 are
scanned from rotating device copies (>= 256 MiB in all) so that every step's input comes from HBM; inputs under
16 MiB get the L2 flushed between steps instead.
After the timed regions every rank compares its full record arrays (device-resident and end to end)
with the oracle's scan of the same bytes: `parity` in the line, exit code 1 if they differ.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pfac_synth as synth  # noqa: E402  (workload generators: a tools library, not the product)

WORKLOADS = {
    # name: (pattern kind, count, seed, min_len, max_len, text kind, text seed, default bytes, description)
    "config2": (0, 1000, 1, 8, 32, 0, 2, 256 << 20,
                "config2: 1,000 synthetic patterns (len 8-32) over 256 MiB printable text with planted matches"),
    "config3": (1, 10000, 3, 4, 64, 1, 4, 1 << 30,
                "config3: 10,000 synthetic Snort-like patterns over 1 GiB HTTP-like text per GPU"),
    "config4": (0, 100000, 5, 8, 32, 0, 6, 512 << 20,
                "config4: 100,000 synthetic patterns (len 8-32) over 512 MiB printable text per GPU"),
}
# the reference's own fixtures (tests/golden): pattern file x its 1M text; md5 of GPU_match_result.txt (SURVEY 8c)
FIXTURES = {
    "config1": ("experimentpattern", "c20fe75d264cdcfcc219b1b437ab9267",
                "config1: the reference's experimentpattern over its 1M text (1,048,575 bytes scanned)"),
    "dictionary": ("dictionary", "4f9afaba328ea6d5cf43d76b52c38ab7",
                   "dictionary: the reference's xaa..xad (7,989 words) over its 1M text (1,048,575 bytes scanned)"),
}


ALL_CPUS = os.sched_getaffinity(0)   # before any NUMA binding


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config3", choices=sorted(WORKLOADS) + sorted(FIXTURES))
    ap.add_argument("--bytes", type=int, default=0, help="bytes per rank (weak) or in total (strong); default: the workload's size")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--streams", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-job", action="store_true", help="skip the pfac_job_run leg (N>1, rank 0 over all devices)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the end-to-end leg (default min(steps, 10))")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the records of the last timed step (rank 0) as DIR/*.npy, see dump_outputs()")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        # the reference arm scans a sample whose size comes from a timing calibration: not the same bytes every run
        ap.error("--dump-outputs applies to --impl ours")
    return args


DUMP_MAX_RECORDS = 2_000_000     # 3 float64 arrays of this length: 48 MB, under the 64 MB the dump may take


def dump_outputs(out_dir, records):
    """Writes what a caller of the timed path receives, the (pos, id) records of one scan, so that two builds can be
    compared output for output: count.npy (the number of records), pos.npy and id.npy (float64, exact for 32-bit
    values), and rows.npy, the record numbers pos/id hold -- all records up to DUMP_MAX_RECORDS, beyond that a fixed
    seeded sample of them in record order.  Positions are as the records hold them, relative to the start of the
    dumping rank's shard (rank 0's starts at 0)."""
    n = len(records)
    if n <= DUMP_MAX_RECORDS:
        rows = np.arange(n)
    else:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_RECORDS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    out = {"count": np.array([n], dtype=np.float64), "rows": rows.astype(np.float64),
           "pos": (records[rows, 0].astype(np.int64) & 0xFFFFFFFF).astype(np.float64),   # uint32 held in an int32
           "id": records[rows, 1].astype(np.float64)}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_patterns(name):
    """-> (pattern file image, description, bytes, fixture text or None, golden md5 or None)."""
    if name in FIXTURES:
        from conftest import load_fixtures
        fx = load_fixtures()
        key, md5, desc = FIXTURES[name]
        text = np.frombuffer(fx["1M"], dtype=np.uint8)
        return fx[key], desc, len(text) - 1, text, md5          # the CLI drops the file's last byte (main.cc:138)
    pk, cnt, pseed, lo, hi, tk, tseed, nbytes, desc = WORKLOADS[name]
    return synth.synth_patterns(pk, cnt, pseed, lo, hi), desc, nbytes, None, None


def shard_text(args, pats, mpl, rank, world, n, fixture, out):
    """Fills `out` with rank `rank`'s shard: its start positions followed by its halo (the first
    max_pat_len-1 bytes of the next shard, nothing after the last).  Weak scaling: every rank has its own
    seeded text of n bytes; strong scaling: ONE seeded text of the workload's size, cut by the product's
    sharding rule (pfac_job_plan).  Returns (n_starts, n_valid, base position)."""
    import phfpfac_b200 as pf
    halo = max(mpl - 1, 0)
    if fixture is not None:            # the reference's 1M text (tiled when --bytes asks for more)
        reps = -(-n // len(fixture))
        out[:n] = np.tile(fixture, reps)[:n] if reps > 1 else fixture[:n]
        out[n:] = 0
        return n, n, 0
    tk, tseed = WORKLOADS[args.workload][5], WORKLOADS[args.workload][6]
    if args.scaling == "strong":
        total = args.bytes or WORKLOADS[args.workload][7]
        start, ns, nv = pf.plan_shard(total, world, mpl, rank)
        # the generator works in 64 KiB blocks seeded by their index and shards start on 64 KiB boundaries
        whole = synth.synth_text(tk, tseed, min(total, start + nv), patterns=pats)
        out[:nv] = whole[start:start + nv]
        out[nv:] = 0
        return ns, nv, start
    synth.synth_text(tk, tseed + 1000 * rank, n, patterns=pats, out=out[:n])
    if rank + 1 < world and halo:
        out[n:] = synth.synth_text(tk, tseed + 1000 * (rank + 1), min(n, 65536), patterns=pats)[:halo]
        return n, n + halo, rank * n
    out[n:] = 0
    return n, n, rank * n


def bind_to_gpu_numa_node(index):
    """Best effort: run this rank (and first-touch its pinned buffers) on the NUMA node its GPU hangs
    off, so that eight ranks do not pull their H2D traffic across the socket interconnect."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:       # 00000000:1B:00.0 -> 0000:1b:00.0
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed regions run."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self.active = threading.Event()
        self.period = float(os.environ.get("PFAC_BENCH_SAMPLE_MS", "1")) * 1e-3
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop.is_set():
            if self.active.is_set():
                try:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(self.period)

    def stop(self):
        self._stop.set()

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------- CPU legs (oracle)

def cpu_scan(part, mpl, text, cores, count_only):
    """The oracle's OpenMP port of SUBSEG_MATCH over canonical PHF arrays.  count_only: no records (the
    calibration runs); otherwise ONE pass over the input that writes the (pos, id) records."""
    from _oracle import scan_tables_cpu, scan_tables_cpu_1pass
    if count_only:
        return scan_tables_cpu(part, part.idmap, mpl, text, nthreads=cores, count_only=True)
    return scan_tables_cpu_1pass(part, part.idmap, mpl, text, nthreads=cores)


def host_cores():
    from _oracle import oracle_lib
    # torchrun sets OMP_NUM_THREADS=1 for its workers: take the cores this process may run on instead
    return max(oracle_lib().oracle_max_threads(), len(os.sched_getaffinity(0)))


def bounded_sample(text, rate_bytes_per_s, budget_s):
    sample = int(min(len(text), max(1 << 20, rate_bytes_per_s * budget_s)))
    if sample >= 1 << 20:
        sample &= ~0xFFFFF
    return min(max(sample, min(len(text), 1 << 20)), len(text))


def cpu_baseline(part, mpl, text, budget_s=12.0):
    """The oracle's port of SUBSEG_MATCH over the SAME PHF arrays on host threads (the reference
    ships no CPU matcher, main.cc:239).  Bounded sample: calibrate on 4 MiB, then ~budget_s of work."""
    cores = host_cores()
    cal = min(len(text), 4 << 20)
    t0 = time.perf_counter()
    cpu_scan(part, mpl, text[:cal], cores, True)
    dt = max(time.perf_counter() - t0, 1e-6)
    sample = bounded_sample(text, cal / dt, budget_s)
    best, cnt = None, 0
    for _ in range(2):
        t0 = time.perf_counter()
        pos, _ids = cpu_scan(part, mpl, text[:sample], cores, False)
        dt = time.perf_counter() - t0
        cnt = len(pos)
        best = dt if best is None else min(best, dt)
    return {"value": sample / best / 1e9, "unit": "GB/s", "cores": cores, "kind": "port",
            "sample": f"first {sample} bytes of the rank-0 shard, best of 2, {cnt} records written"}


def shared_config(args, desc, nbytes, fixture, world):
    """The `config` object of BOTH arms (the driver compares them): a pure function of the command line and
    the workload.  What a run finds out (match counts, table sizes, the L2 handling it chose) goes into the
    line's `detail` object instead."""
    strong = args.scaling == "strong" and fixture is None
    if strong:
        total = args.bytes or nbytes
        per = min(total, (-(-total // world) + 65535) & ~65535)   # pfac_job_plan's rule: shard 0 of `world`
    else:
        per = args.bytes or nbytes
        total = per * world
    if per >= (192 << 20):
        l2 = "input per step exceeds the 126 MB L2; no flush needed"
    elif per >= (16 << 20):
        l2 = ("input smaller than the L2: the steps rotate over device copies of the shard that together exceed "
              "256 MiB, so every step's input comes from HBM")
    else:
        l2 = "input fits the L2: a 256 MiB buffer is written between timed steps, every step timed by its own event pair"
    return {"workload": desc, "bytes_per_gpu": per, "streams_per_gpu": args.streams, "phf_width": 256,
            "scaling": args.scaling, "total_bytes": total, "l2": l2,
            "timed": "value: input resident in HBM; e2e: host buffers, H2D and D2H inside the timed region",
            "parallelism": f"input sharded x{world} ({args.scaling}), no collective"}


def run_reference(args):
    """The reference arm: the reference's scan on the box's host cores.  The reference ships no CPU
    matcher (main.cc only ever calls GPU_TraceTable) and its kernel does not build on CUDA 12, so this
    is the oracle's OpenMP port of SUBSEG_MATCH over tables built by the oracle's restatement of
    CreateTable + FFDM.  Hermetic: neither the product library nor its Python package is loaded."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from _oracle import Oracle
    pats, desc, nbytes, fixture, _ = workload_patterns(args.workload)
    n = args.bytes or nbytes
    o = Oracle(pats, n_parts=1, width=256)
    part, mpl = o.part(0), o.max_pat_len
    cores = host_cores()
    if fixture is not None:
        text = fixture[:n]
    else:
        tk, tseed = WORKLOADS[args.workload][5], WORKLOADS[args.workload][6]
        text = synth.synth_text(tk, tseed, min(n, 256 << 20), patterns=pats)
    # bounded sample per step so K+W steps end within a few minutes
    cal_n = min(len(text), 4 << 20)
    t0 = time.perf_counter()
    cpu_scan(part, mpl, text[:cal_n], cores, True)
    rate = cal_n / max(time.perf_counter() - t0, 1e-6)
    sample = bounded_sample(text, rate, 120.0 / max(args.steps + args.warmup, 1))
    n_rec = 0
    for _ in range(args.warmup):
        cpu_scan(part, mpl, text[:sample], cores, False)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pos, _ids = cpu_scan(part, mpl, text[:sample], cores, False)     # records written, like the product
        n_rec = len(pos)
    dt = time.perf_counter() - t0
    v = sample * args.steps / dt / 1e9
    cfg = shared_config(args, desc, nbytes, fixture, int(os.environ.get("WORLD_SIZE", "1")))
    line = {
        "impl": "reference", "metric": "input GB/s matched", "value": v, "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "u8", "data": "synthetic" if fixture is None else "reference fixture",
        "config": cfg,
        "cpu_baseline": {"value": v, "unit": "GB/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} bytes of the rank-0 shard per step, {n_rec} records written"},
        "e2e": {"value": v, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": ("the reference ships no CPU matcher and its kernel does not compile on CUDA 12; this arm is the "
                 "oracle's OpenMP port of SUBSEG_MATCH over the oracle-built PHF tables, records written"),
    }
    line["reference_gpu"] = reference_gpu_leg(args)
    print(json.dumps(line))
    return 0


def reference_gpu_leg(args):
    """Context for the reference arm: the reference's own GPU path (master_kernel.cu built for
    sm_100a, oracle/_ref) on the largest input its 32-bit dense result can index, in a subprocess.
    Reported beside the CPU number, never instead of it; None where it cannot run."""
    import re
    import subprocess
    tool = os.path.join(ROOT, "tests", "refgpu_bench.py")
    so = os.path.join(ROOT, "oracle", "_ref", "libphfpfac_refgpu.so")
    try:
        import torch
        if not (os.path.exists(tool) and os.path.exists(so) and torch.cuda.is_available()):
            return None
        r = subprocess.run([sys.executable, tool, "--workload", args.workload, "--no-compare"], capture_output=True,
                           text=True, timeout=150)
        if r.returncode != 0:
            return None
        out = json.loads(r.stdout.strip().splitlines()[-1])
        k = re.findall(r"2\. MASTER: The elapsed time is ([0-9.]+) ms", r.stdout)
        kernel_ms = min(float(x) for x in k) if k else None
        return {"bytes": out["bytes"], "kernel_ms": kernel_ms,
                "kernel_gbs": out["bytes"] / kernel_ms / 1e6 if kernel_ms else None,
                "end_to_end_ms": sum(v for v in (out["ms"]["malloc_memset"], out["ms"]["trace_h2d_kernel_d2h"], out["ms"]["free"])),
                "h2d_kernel_d2h_ms": out["ms"]["trace_h2d_kernel_d2h"],
                "end_to_end_gbs": out["gbs_end_to_end"],
                "note": "GPU_Malloc_Memory + GPU_TraceTable + GPU_Free_memory of master_kernel.cu (tex1Dfetch -> __ldg), "
                        "dense result of 4*max_pat_len bytes per input byte copied back; host-side sift not included"}
    except Exception:
        return None


# --------------------------------------------------------------------------------- the product arm

def job_leg_rank0(args, pf, torch, tables, pats, part, mpl, world, n_per_gpu):
    """The product's own multi-GPU scheduler (pfac_job_run: one host thread per GPU, shard + halo per GPU,
    stream pipeline per GPU), driven from ONE process over all N devices."""
    tk, tseed = WORKLOADS[args.workload][5], WORKLOADS[args.workload][6]
    total = n_per_gpu * world
    # this process was bound to GPU 0's NUMA node for the per-rank legs; the job feeds every GPU from one
    # buffer, so its pages are first-touched (by the generator's threads) from all the CPUs again
    try:
        os.sched_setaffinity(0, ALL_CPUS)
    except Exception:
        pass
    big = torch.empty(total, dtype=torch.uint8, pin_memory=True)
    synth.synth_text(tk, tseed + 7, total, patterns=pats, out=big.numpy())
    job = pf.Job(tables, devices=list(range(world)), streams_per_gpu=args.streams)
    job.run(big.numpy())                     # warm-up: contexts, buffers
    best, nm, segs = None, 0, []
    for _ in range(3):
        t0 = time.perf_counter()
        nm, segs = job.run(big.numpy())
        dtj = time.perf_counter() - t0
        best = dtj if best is None else min(best, dtj)
    # check: the job's records against the oracle on the first and the last GPU's shard
    ok = True
    for g in sorted({0, world - 1}):
        s0, ns, nv = pf.plan_shard(total, world, mpl, g)
        p_, i_ = cpu_scan(part, mpl, big.numpy()[s0:s0 + nv], host_cores(), False)
        k_ = p_ < ns
        mine = [(b, a) for b, a in segs if s0 <= b < s0 + ns and len(a)]
        gp = np.concatenate([a[:, 0].astype(np.int64) + b for b, a in mine] or [np.zeros(0, np.int64)])
        gi = np.concatenate([a[:, 1].astype(np.int64) for b, a in mine] or [np.zeros(0, np.int64)])
        ok = ok and np.array_equal(gp, p_[k_] + s0) and np.array_equal(gi, i_[k_].astype(np.int64))
    job.close()
    return {"value": total / best / 1e9, "unit": "GB/s", "devices": world, "bytes": total, "matches": int(nm),
            "best_of": 3, "records_equal_oracle_on_first_and_last_shard": bool(ok),
            "note": "pfac_job_run from ONE process over all devices (pinned host input, H2D, scan, D2H), wall clock"}


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    import torch
    import phfpfac_b200 as pf
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the PFAC scan has no CPU path")
    torch.cuda.set_device(local_rank)
    numa_node = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pats, desc, nbytes, fixture, golden_md5 = workload_patterns(args.workload)
    tables = pf.Tables.from_bytes(pats, n_parts=1, width=256)
    mpl = tables.max_pat_len
    halo = mpl - 1
    strong = args.scaling == "strong" and fixture is None
    if strong:
        total_bytes = args.bytes or nbytes
        n = pf.plan_shard(total_bytes, world, mpl, rank)[1]
    else:
        n = args.bytes or nbytes
        total_bytes = n * world
    # the rank's shard in pinned host memory, followed by the halo = first bytes of the next shard
    h_text = torch.empty(n + halo, dtype=torch.uint8, pin_memory=True)
    text = h_text.numpy()
    n, n_valid, base_pos = shard_text(args, pats, mpl, rank, world, n, fixture, text)
    d_text = h_text.cuda()
    m = pf.Matcher(tables, device=local_rank, n_streams=args.streams, chunk_bytes=0)
    cap = max(n // 8, 1 << 16)
    d_out = torch.empty((cap, 2), dtype=torch.int32, device="cuda")
    d_cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    # a real (non-default) stream: handle 0 would mean "the library's own stream" to the C ABI, and
    # torch.cuda.Event must be recorded on the stream the kernel runs on
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    # Inputs smaller than the 126 MB L2 must not be re-read from it step after step.  From 16 MiB up the step
    # rotates over copies of the shard that together exceed twice the L2 (the input of every step comes from
    # HBM, the tables stay warm -- what a GPU sees when it scans fresh data each time); smaller inputs get the
    # L2 flushed between steps (below).
    d_copies = [d_text]
    if (16 << 20) <= n < (192 << 20):
        while len(d_copies) * (n + halo) < (256 << 20) + (n + halo):
            d_copies.append(d_text.clone())
    step_no = [0]

    def step_dev():
        d = d_copies[step_no[0] % len(d_copies)]
        step_no[0] += 1
        m.scan_device_raw(d.data_ptr(), n, n_valid, base_pos, d_out.data_ptr(), cap, d_cnt.data_ptr(), stream)

    sampler = ClockSampler(local_rank)
    sampler.start()
    step_dev()
    torch.cuda.synchronize()
    n_matches = int(d_cnt.item())
    if n_matches > cap:      # dense workload: size the record buffer to what the scan reports
        cap = n_matches
        d_out = torch.empty((cap, 2), dtype=torch.int32, device="cuda")
    for _ in range(max(args.warmup, 3)):
        step_dev()
    torch.cuda.synchronize()
    n_matches = int(d_cnt.item())
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    # small inputs fit the 126 MB L2: flush it between timed steps (write a buffer larger than L2) and time
    # every step with its own event pair
    flush = n < (16 << 20)
    d_flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if flush else None
    sampler.active.set()

    def timed_steps():
        if flush:
            t = 0.0
            for _ in range(args.steps):
                d_flush.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                step_dev()
                e1.record()
                torch.cuda.synchronize()
                t += e0.elapsed_time(e1)
            return t
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(args.steps):
            step_dev()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1)

    ms = timed_steps()      # the bench value: exactly args.steps steps, nothing between the kernels of a step
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_out[:int(d_cnt.item())].cpu().numpy())
    # the roofline's kernel time: the same steps once more with an event pair around the dominant kernel of every
    # launch sequence, on its stream (the pair sits between the kernels of a step, so these steps are not the value)
    m.set_timing(True)
    timed_steps()
    sampler.active.clear()
    kernel_ms_total, kernel_launches = m.kernel_time()
    m.set_timing(False)
    warm = None
    if flush:
        # the same steps back to back with a warm L2 and no event pair around each kernel: NOT the bench value
        # (the input fits the L2), reported because the reference's own kernel time -- one launch right after
        # its H2D copy, `reference_gpu` of the reference arm -- is a warm-L2 figure too
        for _ in range(3):
            step_dev()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(max(args.steps, 20)):
            step_dev()
        ev1.record()
        torch.cuda.synchronize()
        warm_ms = ev0.elapsed_time(ev1) / max(args.steps, 20)
        warm = {"ms_per_step": warm_ms, "value": n / (warm_ms * 1e-3) / 1e9, "unit": "GB/s",
                "note": "steps back to back, input and tables L2-resident (the input is smaller than the L2): like for like with "
                        "reference_gpu.kernel_ms of `bench.py --impl reference`, which is one launch right after its H2D copy"}
    dev_records = d_out[:n_matches].cpu().numpy().copy()
    dev_launches_per_step = m.last_info()["launches"]
    if dist:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        ms_max = float(t.item())
    else:
        ms_max = ms
    torch.cuda.synchronize()
    launches = dev_launches_per_step * args.steps

    # ---- end to end through the public host API: pinned input -> H2D -> scan -> D2H records
    e2e_steps = args.e2e_steps or min(args.steps, 10)
    h_out = torch.empty((cap, 2), dtype=torch.int32, pin_memory=True)
    cnt = C.c_uint64(0)

    def step_e2e():
        pf.check(pf.lib.pfac_scan_host(m._h, h_text.data_ptr(), n, n_valid, base_pos, h_out.data_ptr(), cap,
                                       C.byref(cnt)))

    for _ in range(2):
        step_e2e()
    assert cnt.value == n_matches, (cnt.value, n_matches)
    if dist:
        dist.barrier()
    sampler.active.set()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    e2e_s = time.perf_counter() - t0
    sampler.active.clear()
    info = m.last_info()
    e2e_records = h_out[:n_matches].numpy().copy()
    if dist:
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
        tm = torch.tensor([n_matches], dtype=torch.int64, device="cuda")
        dist.all_reduce(tm)
        total_matches = int(tm.item())
    else:
        total_matches = n_matches
    sampler.stop()
    launches_e2e = info["launches"] * e2e_steps

    # ---- the ceiling of the e2e leg: bare H2D copies of the same pinned buffers -- one rank alone (rank 0)
    # and all ranks at once (what the host's PCIe fabric gives N GPUs together)
    link_gbs = None
    if rank == 0:
        best = None
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            d_text.copy_(h_text, non_blocking=True)
            e1.record()
            torch.cuda.synchronize()
            best = e0.elapsed_time(e1) if best is None else min(best, e0.elapsed_time(e1))
        link_gbs = h_text.numel() / best / 1e6
    concurrent_gbs = None
    if dist:
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            d_text.copy_(h_text, non_blocking=True)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / 3
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tb = torch.tensor([float(h_text.numel())], dtype=torch.float64, device="cuda")
        dist.all_reduce(tb)
        concurrent_gbs = float(tb.item()) / float(t.item()) / 1e9
        dist.barrier()

    # ---- parity, outside the timed regions: the FULL record arrays against the oracle's scan of this
    # rank's bytes over the SAME canonical tables (every rank; AND-reduced)
    part = tables.part(0)
    cores = host_cores() if world == 1 else max(1, host_cores() // world)
    opos, oids = cpu_scan(part, mpl, text[:n_valid], cores, False)
    keep = opos < n
    opos, oids = opos[keep], oids[keep]

    def same(rec):
        return bool(len(rec) == len(opos) and np.array_equal(rec[:, 0].astype(np.int64) & 0xFFFFFFFF, opos)
                    and np.array_equal(rec[:, 1].astype(np.int64), oids.astype(np.int64)))

    equal_dev, equal_e2e = same(dev_records), same(e2e_records)
    result_md5 = None
    if golden_md5 is not None and world == 1 and not args.bytes:
        rec = np.zeros(len(e2e_records), dtype=pf.MATCH_DTYPE)
        rec["pos"], rec["id"] = e2e_records[:, 0], e2e_records[:, 1]
        result_md5 = hashlib.md5(pf.format_records(rec, base_pos=0)).hexdigest()
    parity_ok = equal_dev and equal_e2e and (result_md5 is None or result_md5 == golden_md5)
    if dist:
        t = torch.tensor([1 if parity_ok else 0], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        parity_all = bool(t.item())
    else:
        parity_all = parity_ok

    job_leg = None
    if dist and not args.no_job and fixture is None:
        if rank == 0:
            try:
                job_leg = job_leg_rank0(args, pf, torch, tables, pats, part, mpl, world,
                                        n if not strong else max(65536, (total_bytes // world) & ~65535))
            except Exception as e:   # never lose the main line to this leg
                job_leg = {"error": str(e)[:300]}
        # The other ranks wait on the HOST (a key of the rendezvous store) until rank 0's job leg is over: in an
        # NCCL barrier they would keep a kernel spinning on their GPUs, which rank 0's job uses from its own process
        try:
            store = dist.distributed_c10d._get_default_store()
            if rank == 0:
                store.set("pfac_job_leg_done", "1")
            else:
                store.wait(["pfac_job_leg_done"])
        except Exception:
            pass
        dist.barrier()

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        plain = not args.bytes and args.scaling == "weak"
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(args.workload if plain else "", None)
        dinfo = m.derived_info()
        dense_first = dev_launches_per_step == 1
        kernel_name = "pfac_dense_kernel<DIRECT>" if dense_first else \
            ("pfac_scan2_kernel" if dinfo["mode"] == 0 else "pfac_scan_kernel")
        ncu = None   # selected metrics of the committed ncu capture of the dominant kernel (not measured in this run)
        npath = os.path.join(ROOT, "profiles", "r2_ncu_detector_config3_1GiB.json")   # tools/ncu_summary.py
        if os.path.exists(npath) and args.workload == "config3" and plain:
            capture = json.load(open(npath))["kernels"][0]

            def _bytes(v):   # "1.074303 Gbyte" -> bytes
                x, u = str(v).split()[:2]
                return float(x) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[u]
            if "dram__bytes_read.sum" in capture and "dram__bytes_write.sum" in capture:
                traffic = _bytes(capture["dram__bytes_read.sum"]) + _bytes(capture["dram__bytes_write.sum"])
            pick = {"smem_pipe_pct_of_peak": "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed",
                    "issue_active_pct": "smsp__issue_active.avg.pct_of_peak_sustained_active",
                    "alu_pipe_pct": "sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active",
                    "dram_pct_of_peak": "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
                    "warp_instructions": "smsp__inst_executed.sum",
                    "shared_wavefronts": "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum",
                    "threads_per_instruction": "smsp__thread_inst_executed_per_inst_executed.ratio"}
            ncu = {k: float(str(capture[v]).split()[0]) for k, v in pick.items() if v in capture}
            ncu["source"] = "profiles/r2_ncu_detector_config3_1GiB.json (ncu --set full, same workload)"
        ms_step = ms_max / args.steps
        alg_bytes = n + 8 * n_matches           # per launch: input bytes + 8 B per match record
        kernel_ms = kernel_ms_total / max(kernel_launches, 1)
        achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
        job_bytes = total_bytes if strong else world * n
        cfg = shared_config(args, desc, nbytes, fixture, world)
        detail = {"matches_per_gpu_step": n_matches, "total_matches": total_matches, "tables": dinfo,
                  "bytes_rank0": n, "device_copies_rotated": len(d_copies), "l2_flushed_between_steps": bool(flush),
                  "numa_node_rank0": numa_node}
        line = {
            "metric": "input GB/s matched", "value": job_bytes * args.steps / (ms_max * 1e-3) / 1e9,
            "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "u8", "data": "synthetic" if fixture is None else "reference fixture",
            "config": cfg, "detail": detail,
            "clocks": sampler.summary(),
            "e2e": {"value": job_bytes * e2e_steps / e2e_s / 1e9, "unit": "GB/s", "steps": e2e_steps,
                    "h2d_bytes_per_step": int(info["h2d_bytes"]), "d2h_bytes_per_step": int(info["d2h_bytes"]),
                    "launches_per_step": int(info["launches"]), "ms_per_step": e2e_s / e2e_steps * 1e3,
                    "h2d_copy_alone_gbs": link_gbs, "h2d_concurrent_gbs_total": concurrent_gbs,
                    "note": "h2d_copy_alone_gbs = a bare cudaMemcpyAsync of rank 0's pinned input alone; "
                            "h2d_concurrent_gbs_total = all ranks copying their pinned shards at the same time "
                            "(the ceiling of this leg at N GPUs), both measured in this run"},
            "gpu_launches": int(world * (launches + launches_e2e)),
            "parity": {"records": int(total_matches), "equal": parity_all,
                       "device_resident_equal_oracle": equal_dev, "e2e_equal_oracle": equal_e2e,
                       "result_md5": result_md5, "golden_md5": golden_md5,
                       "note": "full (pos, id) record arrays of both legs vs the oracle's OpenMP scan of the same bytes, every rank"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "kernel": kernel_name, "ncu": ncu, "algorithmic_bytes_per_launch": alg_bytes,
                         "kernel_ms_per_launch": kernel_ms, "kernel_launches_timed": kernel_launches,
                         "kernel_share_of_step": kernel_ms / (ms / args.steps),
                         "note": "a step = the detector (which also walks the surviving candidates and writes their "
                                 "records) + pfac_dense_kernel (returns at once unless tiles were handed over) + "
                                 "pfac_finalize_kernel; `value` covers all of them, `achieved` the dominant kernel alone"},
        }
        if job_leg is not None:
            line["e2e_job"] = job_leg
        if warm is not None:
            line["warm_l2"] = warm
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(part, mpl, text[:n])
        print(json.dumps(line))
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    m.close()
    return 0 if parity_all else 1


if __name__ == "__main__":
    sys.exit(main())
