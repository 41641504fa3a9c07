"""Batch scan of many independent documents (pfac_scan_batch_device) against its floor and against one call per
document, config-3 patterns.  Prints one JSON line.

  (a) packets:   100,000 documents of 40-1500 bytes cut from the config-3 text
  (b) documents: log-uniform sizes from 64 B to 64 KiB, at least 256 MiB in all (beyond the 126 MB L2)

Per workload, CUDA-event times (warmed, averaged over --reps calls):
  batch_ms   one pfac_scan_batch_device over the packed documents
  packed_ms  one pfac_scan_device over the same bytes (the floor: no split, straddling matches included)
  loop       pfac_scan_device once per document over the first 2,000 documents
Parity: the batch records equal the per-document loop's on those documents, and on the whole batch they equal
the packed scan's records with the matches that run past their document's end dropped (pattern_lengths).

    python tools/batch_bench.py [--reps 20] [--loop-docs 2000]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def workload_sizes(kind, rng):
    if kind == "packets":
        return rng.integers(40, 1501, 100000)
    sizes, total = [], 0
    while total < (256 << 20):
        s = int(np.exp(rng.uniform(np.log(64), np.log(64 << 10))))
        sizes.append(s)
        total += s
    return np.array(sizes)


def timed(torch, stream, fn, reps):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(reps):
        fn()
    ev1.record(stream)
    ev1.synchronize()
    return ev0.elapsed_time(ev1) / reps


def run(kind, pats, lengths, m, args, torch, lib, pf, synth):
    rng = np.random.default_rng({"packets": 101, "documents": 202}[kind])
    sizes = workload_sizes(kind, rng)
    total = int(sizes.sum())
    text = synth.synth_text(1, 4, total + 1, patterns=pats)[:total]   # the documents, back to back
    offs = np.zeros(len(sizes) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum(sizes)
    n_docs = len(sizes)
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    d = torch.from_numpy(text).cuda()
    cap = max(1 << 20, total // 64)
    out = torch.empty((cap, 2), dtype=torch.int32, device="cuda")
    first = torch.empty(n_docs + 1, dtype=torch.int64, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    out2 = torch.empty((cap, 2), dtype=torch.int32, device="cuda")
    cnt2 = torch.zeros(1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()

    def batch():
        pf.check(lib.pfac_scan_batch_device(m._h, d.data_ptr(), offs.ctypes.data, n_docs, out.data_ptr(), cap,
                                            first.data_ptr(), cnt.data_ptr(), sp))

    def packed():
        pf.check(lib.pfac_scan_device(m._h, d.data_ptr(), total, total, 0, out2.data_ptr(), cap, cnt2.data_ptr(), sp))

    n_loop = min(args.loop_docs, n_docs)
    out3 = torch.empty((1 << 16, 2), dtype=torch.int32, device="cuda")
    cnts3 = torch.zeros(n_loop, dtype=torch.int64, device="cuda")
    loop_bytes = int(offs[n_loop])

    def loop():
        for i in range(n_loop):
            a, b = int(offs[i]), int(offs[i + 1])
            pf.check(lib.pfac_scan_device(m._h, d.data_ptr() + a, b - a, b - a, 0, out3.data_ptr(), 1 << 16,
                                          cnts3.data_ptr() + 8 * i, sp))

    for _ in range(3):   # warm-up of every shape the timed windows use
        batch()
        packed()
    loop()
    stream.synchronize()
    batch_ms = timed(torch, stream, batch, args.reps)
    packed_ms = timed(torch, stream, packed, args.reps)
    batch_ms2 = timed(torch, stream, batch, args.reps)   # alternated: a drift of the card shows as batch_ms != batch_ms2
    info = m.last_info()
    loop_ms = timed(torch, stream, loop, 1)

    # parity
    first_h, rec = m.scan_batch(d, offs, cap=cap)
    packed_rec = m.scan_device(d, cap=cap)
    pos = packed_rec["pos"].astype(np.int64)
    doc = np.searchsorted(offs[1:].astype(np.int64), pos, side="right")
    keep = pos + lengths[packed_rec["id"].astype(np.int64)] <= offs[1:].astype(np.int64)[doc]
    want = packed_rec[keep].copy()
    want["pos"] = (pos[keep] - offs[:-1].astype(np.int64)[doc[keep]]).astype(np.uint32)
    parity_packed = bool(np.array_equal(rec, want))
    want_first = np.searchsorted(doc[keep], np.arange(n_docs + 1), side="left").astype(np.uint64)
    parity_packed = parity_packed and bool(np.array_equal(first_h, want_first))
    parity_loop = True
    for i in range(n_loop):
        a, b = int(offs[i]), int(offs[i + 1])
        got = m.scan_device(d, n_starts=b - a, n_valid=b - a, offset=a, cap=1 << 12)
        if not np.array_equal(rec[int(first_h[i]):int(first_h[i + 1])], got):
            parity_loop = False
            break
    per_doc_us = loop_ms * 1e3 / n_loop
    batch_same_bytes_ms = batch_ms * loop_bytes / total
    return {
        "docs": n_docs, "bytes": total, "mean_doc_bytes": round(total / n_docs, 1),
        "records": int(len(rec)), "packed_records": int(len(packed_rec)),
        "batch_ms": round(batch_ms, 4), "batch_ms_repeat": round(batch_ms2, 4), "packed_ms": round(packed_ms, 4),
        "batch_over_packed": round(batch_ms / packed_ms, 3), "batch_minus_packed_us": round((batch_ms - packed_ms) * 1e3, 1),
        "batch_gbs": round(total / batch_ms / 1e6, 1), "packed_gbs": round(total / packed_ms / 1e6, 1),
        "loop": {"docs": n_loop, "bytes": loop_bytes, "ms": round(loop_ms, 3), "us_per_doc": round(per_doc_us, 2),
                 "speedup_at_equal_bytes": round(loop_ms / batch_same_bytes_ms, 1)},
        "launches_per_batch": int(info["launches"]),
        "parity": {"batch_equal_per_document_loop": parity_loop, "batch_equal_filtered_packed_scan": parity_packed},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--loop-docs", type=int, default=2000)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("batch_bench.py measures on the GPU; none is available")
    import phfpfac_b200 as pf
    from phfpfac_b200._lib import lib
    import pfac_synth as synth
    from bench import WORKLOADS

    name, power = card()
    pk, count, pseed, lo, hi = WORKLOADS["config3"][:5]
    pats = synth.synth_patterns(pk, count, pseed, lo, hi)
    t = pf.Tables.from_bytes(pats, 1, 256)
    lengths = t.pattern_lengths()
    m = pf.Matcher(t, device=0)
    res = {"metric": "batch scan of independent documents", "patterns": "config3 (10,000 synthetic Snort-like)",
           "gpu": name, "power_limit": power, "reps": args.reps}
    for kind in ("packets", "documents"):
        res[kind] = run(kind, pats, lengths, m, args, torch, lib, pf, synth)
    res["parity"] = all(all(res[k]["parity"].values()) for k in ("packets", "documents"))
    m.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
