"""Cost of per-pattern case rules (PFAC_PATTERNS_CASE_RULES): a mixed set against the uniform caseless set of the same
config-3 lines.  Every third line (ids 3, 6, 9, ...) is exact, the others caseless.  Both sets have the same automaton,
so the difference is the verify pass (and, for the library's own input, the out-of-place fold).  The mixed arm's
records are checked against the reference (tests/_case_rules_ref.py) in the same run.  Writes
profiles/r6_case_rules_bench.json (or --out) and prints it as one JSON line.

  device      config 3 (10,000 Snort-like patterns, 1 GiB HTTP-like text), device-resident; CUDA events, arms alternating
  packets     100,000 packets of 40-1500 B cut from the same text, one scan_batch
  host        pfac_scan_host of the 1 GiB text from pinned memory (host clock around the synchronous call)
  kernels     the two verify kernels alone: torch.profiler, CUDA activities, in a window of its own
  dictionary  the reference's dictionary fixture (patterns of 1-3+ bytes: nearly every position reports), 16 MiB of
              text: the pass's cost grows with the records

    python tools/case_rules_bench.py [--reps 20] [--host-reps 6] [--out profiles/r6_case_rules_bench.json]
"""
import argparse
import ctypes as C
import gzip
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

from caseless_bench import alternate, card   # noqa: E402


def every_third_exact(n):
    return (np.arange(n) % 3 != 2).astype(np.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--host-reps", type=int, default=6)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_case_rules_bench.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("case_rules_bench.py measures on the GPU; none is available")
    import phfpfac_b200 as pf
    from phfpfac_b200._lib import lib
    import pfac_synth as synth
    from bench import WORKLOADS
    from _case_rules_ref import CaseRulesRef

    name, power = card()
    pk, count, pseed, lo, hi, tk, tseed, nbytes = WORKLOADS["config3"][:8]
    pats = synth.synth_patterns(pk, count, pseed, lo, hi)
    n_pat = pats.count(b"\n")
    rules = every_third_exact(n_pat)
    mixed_t = pf.Tables.from_bytes(pats, 1, 256, caseless=rules)
    mx = pf.Matcher(mixed_t, device=0, n_streams=4)
    ci = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256, caseless=True), device=0, n_streams=4)
    text = synth.synth_text(tk, tseed, nbytes, patterns=pats)
    res = {"metric": "mixed case rules (fold out of place + unchanged scan + verify pass) against the caseless scan "
                     "of the same lines",
           "workload": "config3: 10,000 synthetic Snort-like patterns, 1 GiB HTTP-like text",
           "rules": "every third line exact (ids 3, 6, 9, ...), the others caseless",
           "gpu": name, "power_limit": power, "reps": args.reps}
    ref = CaseRulesRef(pats, rules)
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    d = torch.from_numpy(text).cuda()
    cap = len(text) // 8
    out = [torch.empty((cap, 2), dtype=torch.int32, device="cuda") for _ in range(2)]
    cnt = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(2)]
    torch.cuda.synchronize()

    def dev(m, src, k, c=cap):
        return lambda: pf.check(lib.pfac_scan_device(m._h, src.data_ptr(), src.numel(), src.numel(), 0, out[k].data_ptr(),
                                                     c, cnt[k].data_ptr(), C.c_void_p(sp)))

    def same_as_ref(rec, want):
        return len(rec) == len(want[0]) and np.array_equal(rec[:, 0], want[0]) and np.array_equal(rec[:, 1], want[1])

    # ---- device-resident, 1 GiB
    t = alternate(torch, stream, {"mixed": dev(mx, d, 0), "caseless": dev(ci, d, 1)}, args.reps)
    stream.synchronize()
    n = int(cnt[0].item())
    want = ref.scan(text)
    parity_dev = n <= cap and same_as_ref(out[0][:n].cpu().numpy().astype(np.int64), want)
    res["device"] = {"bytes": len(text), "records_mixed": n, "records_caseless": int(cnt[1].item()),
                     "mixed_ms": t["mixed"], "caseless_ms": t["caseless"], "cost_us": (t["mixed"] - t["caseless"]) * 1e3,
                     "ratio": t["mixed"] / t["caseless"], "parity": parity_dev}
    mx.scan_device(d[:1 << 20])
    ci.scan_device(d[:1 << 20])
    res["device"]["launches_mixed"] = mx.last_info()["launches"]
    res["device"]["launches_caseless"] = ci.last_info()["launches"]

    # ---- the verify kernels alone (torch.profiler).  A programmatic dependent launch starts before the kernel
    # ahead of it ends and waits for it, so its profiled time includes that wait; a context created with
    # PFAC_NO_PDL=1 launches in plain stream order, and its kernel times are their own.
    from torch.profiler import ProfilerActivity, profile
    os.environ["PFAC_NO_PDL"] = "1"
    plain = pf.Matcher(mixed_t, device=0, n_streams=4)
    del os.environ["PFAC_NO_PDL"]
    res["kernels"] = {}
    for key, m in (("pdl", mx), ("plain_stream_order", plain)):
        dev(m, d, 0)()
        stream.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                dev(m, d, 0)()
            stream.synchronize()
        kern = {}
        for k in prof.key_averages():
            for kn in ("pfac_rules_count_kernel", "pfac_rules_write_kernel", "pfac_fold_kernel", "pfac_finalize_kernel"):
                if kn in k.key:
                    us = getattr(k, "device_time_total", getattr(k, "cuda_time_total", 0.0))
                    kern[kn] = {"launches": k.count, "us_per_launch": us / k.count if k.count else float("nan")}
        res["kernels"][key] = kern
    plain.close()

    # ---- 100,000 packets of 40-1500 B
    rng = np.random.default_rng(101)
    sizes = rng.integers(40, 1501, 100000)
    offs = np.zeros(len(sizes) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum(sizes)
    total = int(offs[-1])
    pk_d = d[:total]
    bcap = max(1 << 20, total // 8)
    bout = [torch.empty((bcap, 2), dtype=torch.int32, device="cuda") for _ in range(2)]
    bfirst = [torch.empty(len(sizes) + 1, dtype=torch.int64, device="cuda") for _ in range(2)]

    def batch(m, k):
        return lambda: pf.check(lib.pfac_scan_batch_device(m._h, pk_d.data_ptr(), offs.ctypes.data, len(sizes),
                                                           bout[k].data_ptr(), bcap, bfirst[k].data_ptr(),
                                                           cnt[k].data_ptr(), C.c_void_p(sp)))
    t = alternate(torch, stream, {"mixed": batch(mx, 0), "caseless": batch(ci, 1)}, args.reps)
    stream.synchronize()
    n = int(cnt[0].item())
    first = bfirst[0].cpu().numpy()
    rec = bout[0][:n].cpu().numpy().astype(np.int64)
    parity_b = n <= bcap
    for i in rng.integers(0, len(sizes), 300).tolist():   # 300 packets against the reference
        a, b = int(offs[i]), int(offs[i + 1])
        parity_b = parity_b and same_as_ref(rec[int(first[i]):int(first[i + 1])], ref.scan(text[a:b]))
    res["packets"] = {"docs": len(sizes), "bytes": total, "records_mixed": n, "mixed_ms": t["mixed"],
                      "caseless_ms": t["caseless"], "cost_us": (t["mixed"] - t["caseless"]) * 1e3,
                      "ratio": t["mixed"] / t["caseless"], "parity_300_docs": bool(parity_b)}
    del out, bout

    # ---- pfac_scan_host, end to end from pinned memory
    hp = torch.from_numpy(text).pin_memory()
    hcap = len(text) // 8
    hout = [np.zeros(hcap, dtype=pf.MATCH_DTYPE) for _ in range(2)]
    hc = [C.c_uint64(0), C.c_uint64(0)]

    def host(m, k):
        def run():
            t0 = time.perf_counter()
            pf.check(lib.pfac_scan_host(m._h, hp.data_ptr(), len(text), len(text), 0, hout[k].ctypes.data, hcap,
                                        C.byref(hc[k])))
            return time.perf_counter() - t0
        return run
    arms = {"mixed": host(mx, 0), "caseless": host(ci, 1)}
    for fn in arms.values():
        fn()
    acc = {k: [] for k in arms}
    for _ in range(args.host_reps):
        for k, fn in arms.items():
            acc[k].append(fn() * 1e3)
    hm, hcl = float(np.median(acc["mixed"])), float(np.median(acc["caseless"]))
    nh = hc[0].value
    hrec = np.stack([hout[0]["pos"][:nh], hout[0]["id"][:nh]], axis=1).astype(np.int64)
    parity_h = same_as_ref(hrec, want)
    res["host"] = {"bytes": len(text), "records_mixed": nh, "mixed_ms": hm, "caseless_ms": hcl, "ratio": hm / hcl,
                   "mixed_GBps": len(text) / hm / 1e6, "caseless_GBps": len(text) / hcl / 1e6, "parity": parity_h}
    mx.close()
    ci.close()
    del d

    # ---- the dictionary fixture: nearly every position reports
    dpats = gzip.decompress(open(os.path.join(ROOT, "tests", "golden", "dictionary.txt.gz"), "rb").read())
    drules = every_third_exact(dpats.count(b"\n"))
    dmx = pf.Matcher(pf.Tables.from_bytes(dpats, 1, 256, caseless=drules), device=0)
    dci = pf.Matcher(pf.Tables.from_bytes(dpats, 1, 256, caseless=True), device=0)
    dtext = synth.synth_text(tk, tseed, 16 << 20, patterns=dpats)
    dd = torch.from_numpy(dtext).cuda()
    dcap = 4 * len(dtext)
    out = [torch.empty((dcap, 2), dtype=torch.int32, device="cuda") for _ in range(2)]
    torch.cuda.synchronize()
    t = alternate(torch, stream, {"mixed": dev(dmx, dd, 0, dcap), "caseless": dev(dci, dd, 1, dcap)}, max(2, args.reps // 4))
    stream.synchronize()
    n = int(cnt[0].item())
    parity_d = n <= dcap and same_as_ref(out[0][:n].cpu().numpy().astype(np.int64), CaseRulesRef(dpats, drules).scan(dtext))
    res["dictionary"] = {"bytes": len(dtext), "records_mixed": n, "records_caseless": int(cnt[1].item()),
                         "mixed_ms": t["mixed"], "caseless_ms": t["caseless"],
                         "cost_us": (t["mixed"] - t["caseless"]) * 1e3,
                         "cost_ns_per_record": (t["mixed"] - t["caseless"]) * 1e6 / max(n, 1), "parity": parity_d}
    dmx.close()
    dci.close()
    res["parity"] = bool(parity_dev and parity_b and parity_h and parity_d)
    line = json.dumps(res)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    print(line)
    if not res["parity"]:
        sys.exit("the mixed set's records differ from the reference")


if __name__ == "__main__":
    main()
