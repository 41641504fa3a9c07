"""Cost of caseless matching (PFAC_PATTERNS_CASELESS): the device fold before the scan, measured against the
case-sensitive scan of the pre-folded text with the tables of the folded patterns.  The records of the two arms are
equal by definition (and asserted here), so the difference between them is the fold alone.  Writes
profiles/r5_caseless_bench.json (or --out) and prints it as one JSON line.

  device    config 3 (10,000 Snort-like patterns, 1 GiB HTTP-like text), device-resident: the caseless scan of T
            (fold into the context's copy, then the scan) against the case-sensitive scan of fold(T); CUDA events,
            the arms alternating
  kernel    pfac_fold_kernel alone (torch.profiler, CUDA activities, in a window of its own) against a bare
            device-to-device cudaMemcpyAsync of the same bytes (CUDA events): both read and write the input once
  packets   100,000 packets of 40-1500 B cut from the same text, one scan_batch (L2-resident)
  host      pfac_scan_host of the 1 GiB text from pinned memory, end to end (host clock around the synchronous call)

    python tools/caseless_bench.py [--reps 20] [--host-reps 6] [--out profiles/r5_caseless_bench.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

FOLD = np.array([b + 0x20 if 0x41 <= b <= 0x5A else b for b in range(256)], dtype=np.uint8)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def event_ms(torch, stream, fn, reps):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(reps):
        fn()
    ev1.record(stream)
    ev1.synchronize()
    return ev0.elapsed_time(ev1) / reps


def alternate(torch, stream, arms, reps, rounds=5):
    """{arm: mean ms}: the arms timed in turn, `rounds` times, `reps` calls per timing (one warm-up call each)."""
    acc = {k: [] for k in arms}
    for fn in arms.values():
        fn()
    for _ in range(rounds):
        for k, fn in arms.items():
            acc[k].append(event_ms(torch, stream, fn, reps))
    return {k: float(np.median(v)) for k, v in acc.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--host-reps", type=int, default=6)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_caseless_bench.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("caseless_bench.py measures on the GPU; none is available")
    import phfpfac_b200 as pf
    from phfpfac_b200._lib import lib
    import pfac_synth as synth
    from bench import WORKLOADS

    name, power = card()
    pk, count, pseed, lo, hi, tk, tseed, nbytes = WORKLOADS["config3"][:8]
    pats = synth.synth_patterns(pk, count, pseed, lo, hi)
    fpats = FOLD[np.frombuffer(pats, dtype=np.uint8)].tobytes()
    ci = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256, caseless=True), device=0, n_streams=4)
    cs = pf.Matcher(pf.Tables.from_bytes(fpats, 1, 256), device=0, n_streams=4)
    text = synth.synth_text(tk, tseed, nbytes, patterns=pats)
    ftext = FOLD[text]
    res = {"metric": "caseless scan (device fold + unchanged scan) against the case-sensitive scan of the folded text",
           "workload": "config3: 10,000 synthetic Snort-like patterns, 1 GiB HTTP-like text",
           "gpu": name, "power_limit": power, "reps": args.reps,
           "upper_case_share_of_text": round(float(np.count_nonzero((text >= 0x41) & (text <= 0x5A))) / len(text), 4)}
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    d, fd = torch.from_numpy(text).cuda(), torch.from_numpy(ftext).cuda()
    cap = len(text) // 8
    out = [torch.empty((cap, 2), dtype=torch.int32, device="cuda") for _ in range(2)]
    cnt = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(2)]
    torch.cuda.synchronize()

    def dev(m, src, k):
        return lambda: pf.check(lib.pfac_scan_device(m._h, src.data_ptr(), src.numel(), src.numel(), 0, out[k].data_ptr(),
                                                     cap, cnt[k].data_ptr(), C.c_void_p(sp)))

    # ---- device-resident, 1 GiB
    t = alternate(torch, stream, {"caseless": dev(ci, d, 0), "folded": dev(cs, fd, 1)}, args.reps)
    stream.synchronize()
    n = int(cnt[0].item())
    parity_dev = n == int(cnt[1].item()) and n <= cap and torch.equal(out[0][:n], out[1][:n])
    res["device"] = {"bytes": len(text), "matches": n, "caseless_ms": t["caseless"], "folded_ms": t["folded"],
                     "fold_cost_ms": t["caseless"] - t["folded"], "ratio": t["caseless"] / t["folded"],
                     "caseless_GBps": len(text) / t["caseless"] / 1e6, "folded_GBps": len(text) / t["folded"] / 1e6,
                     "launches_caseless": None, "parity": parity_dev}
    ci.scan_device(d[:1 << 20])
    res["device"]["launches_caseless"] = ci.last_info()["launches"]

    # ---- the fold kernel alone (profiler) against a device-to-device copy of the same bytes (events)
    dst = torch.empty_like(d)
    with torch.cuda.stream(stream):
        dst.copy_(d)   # (warm)
        copy_ms = event_ms(torch, stream, lambda: dst.copy_(d), args.reps)
    from torch.profiler import ProfilerActivity, profile
    stream.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.reps):
            dev(ci, d, 0)()
        stream.synchronize()
    fold = [k for k in prof.key_averages() if "pfac_fold_kernel" in k.key]
    fold_n = sum(k.count for k in fold)
    fold_us = sum(getattr(k, "device_time_total", getattr(k, "cuda_time_total", 0.0)) for k in fold)
    fold_ms = fold_us / fold_n / 1e3 if fold_n else float("nan")
    # a fold reads and writes every byte once, like the copy
    res["kernel"] = {"bytes": len(text), "fold_ms": fold_ms, "fold_launches_seen": fold_n,
                     "d2d_copy_ms": copy_ms, "fold_GBps_read_plus_write": 2 * len(text) / fold_ms / 1e6,
                     "copy_GBps_read_plus_write": 2 * len(text) / copy_ms / 1e6,
                     "fold_share_of_copy_rate": copy_ms / fold_ms}
    del dst

    # ---- 100,000 packets of 40-1500 B (L2-resident)
    rng = np.random.default_rng(101)
    sizes = rng.integers(40, 1501, 100000)
    offs = np.zeros(len(sizes) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum(sizes)
    total = int(offs[-1])
    pk_ci, pk_cs = d[:total], fd[:total]
    bcap = max(1 << 20, total // 8)
    bout = [torch.empty((bcap, 2), dtype=torch.int32, device="cuda") for _ in range(2)]
    bfirst = [torch.empty(len(sizes) + 1, dtype=torch.int64, device="cuda") for _ in range(2)]

    def batch(m, src, k):
        return lambda: pf.check(lib.pfac_scan_batch_device(m._h, src.data_ptr(), offs.ctypes.data, len(sizes),
                                                           bout[k].data_ptr(), bcap, bfirst[k].data_ptr(),
                                                           cnt[k].data_ptr(), C.c_void_p(sp)))
    t = alternate(torch, stream, {"caseless": batch(ci, pk_ci, 0), "folded": batch(cs, pk_cs, 1)}, args.reps)
    stream.synchronize()
    n = int(cnt[0].item())
    parity_b = (n == int(cnt[1].item()) and n <= bcap and torch.equal(bout[0][:n], bout[1][:n])
                and torch.equal(bfirst[0], bfirst[1]))
    res["packets"] = {"docs": len(sizes), "bytes": total, "matches": n, "caseless_ms": t["caseless"],
                      "folded_ms": t["folded"], "fold_cost_ms": t["caseless"] - t["folded"],
                      "ratio": t["caseless"] / t["folded"], "parity": parity_b}
    del d, fd, out, bout

    # ---- pfac_scan_host, end to end from pinned memory
    hp = [torch.from_numpy(text).pin_memory(), torch.from_numpy(ftext).pin_memory()]
    hcap = len(text) // 8
    hout = [np.zeros(hcap, dtype=pf.MATCH_DTYPE) for _ in range(2)]
    hc = [C.c_uint64(0), C.c_uint64(0)]

    def host(m, k):
        def run():
            t0 = time.perf_counter()
            pf.check(lib.pfac_scan_host(m._h, hp[k].data_ptr(), len(text), len(text), 0, hout[k].ctypes.data, hcap,
                                        C.byref(hc[k])))
            return time.perf_counter() - t0
        return run
    arms = {"caseless": host(ci, 0), "folded": host(cs, 1)}
    for fn in arms.values():
        fn()
    acc = {k: [] for k in arms}
    for _ in range(args.host_reps):
        for k, fn in arms.items():
            acc[k].append(fn() * 1e3)
    hci, hcs = float(np.median(acc["caseless"])), float(np.median(acc["folded"]))
    nh = hc[0].value
    parity_h = nh == hc[1].value and np.array_equal(hout[0][:nh], hout[1][:nh])
    res["host"] = {"bytes": len(text), "matches": nh, "caseless_ms": hci, "folded_ms": hcs, "ratio": hci / hcs,
                   "caseless_GBps": len(text) / hci / 1e6, "folded_GBps": len(text) / hcs / 1e6, "parity": parity_h}
    res["parity"] = bool(parity_dev and parity_b and parity_h)
    ci.close()
    cs.close()
    line = json.dumps(res)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    print(line)
    if not res["parity"]:
        sys.exit("records differ between the caseless and the folded arm")


if __name__ == "__main__":
    main()
