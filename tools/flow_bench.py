"""Streaming scan of many flows (pfac_scan_flows_device_sync) against the batch scan and the packed scan of the same
bytes, config-3 patterns.  Prints one JSON line.

  (a) packets: 10,000 flows, one packet of 40-1500 B per flow per call, 32 calls
      flows_ms   one pfac_scan_flows_device_sync (synchronous: it includes the read-back of the count)
      batch_ms   pfac_scan_batch_device_sync on the same packets (no carry: straddling matches are lost)
      packed_ms  pfac_scan_device_sync on the packets back to back
  (b) large chunks: 16 flows with 16 MiB chunks (256 MiB per call, beyond the 126 MB L2), 4 calls
      the same three, and the pack kernel alone (torch.profiler, a run of its own) against a bare
      device-to-device cudaMemcpyAsync of the same bytes (CUDA events)
CUDA-event times per call (the calls are synchronous: each time runs from the first enqueue to the host's return),
averaged over the calls after a warm-up pass of every shape.  Parity: every flow's
records over all calls equal one scan of the flow's concatenated bytes (scan_batch of the concatenations for (a),
scan_device per flow for (b)).

    python tools/flow_bench.py [--out profiles/r4_flow_bench.json]
"""
import argparse
import ctypes as C
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


def ev_time(torch, stream, fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1)


def run(kind, m, lengths, pats, torch, pf, lib, synth):
    if kind == "packets":
        n_flows, n_calls = 10000, 32
        rng = np.random.default_rng(303)
        sizes = rng.integers(40, 1501, (n_calls, n_flows))
    else:
        n_flows, n_calls = 16, 4
        sizes = np.full((n_calls, n_flows), 16 << 20, dtype=np.int64)
        rng = np.random.default_rng(404)
    total = int(sizes.sum())
    text = synth.synth_text(1, 4, total + 1, patterns=pats)[:total]
    d_text = torch.from_numpy(text).cuda()
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    per_call = int(sizes.sum(axis=1).max())
    cap = max(1 << 20, per_call // 16)
    out = torch.empty((cap, 2), dtype=torch.int32, device="cuda")
    first = torch.empty(n_flows + 1, dtype=torch.int64, device="cuda")
    cnt = C.c_uint64(0)
    calls = []   # per call: (device offset, chunk offsets, flow ids)
    at = 0
    for c in range(n_calls):
        ids = rng.permutation(n_flows).astype(np.uint32)
        offs = np.zeros(n_flows + 1, dtype=np.uint64)
        offs[1:] = np.cumsum(sizes[c][ids])
        calls.append((at, offs, ids))
        at += int(offs[-1])
    base = np.zeros(n_flows, dtype=np.uint64)

    def flows_call(fs, c, keep=None):
        a, offs, ids = calls[c]
        pf.check(lib.pfac_scan_flows_device_sync(fs._h, d_text.data_ptr() + a, offs.ctypes.data, ids.ctypes.data, n_flows,
                                                 out.data_ptr(), cap, first.data_ptr(), base.ctypes.data, C.byref(cnt), sp))
        if keep is not None:
            n = cnt.value
            fr = first.cpu().numpy()
            chunk = np.repeat(np.arange(n_flows), np.diff(fr))
            rec = out[:n].cpu().numpy().astype(np.int64)
            keep.append((ids[chunk].astype(np.int64), rec[:, 0] + base[chunk].astype(np.int64), rec[:, 1]))

    def batch_call(c):
        a, offs, _ = calls[c]
        pf.check(lib.pfac_scan_batch_device_sync(m._h, d_text.data_ptr() + a, offs.ctypes.data, n_flows, out.data_ptr(),
                                                 cap, first.data_ptr(), C.byref(cnt), sp))

    def packed_call(c):
        a, offs, _ = calls[c]
        n = int(offs[-1])
        pf.check(lib.pfac_scan_device_sync(m._h, d_text.data_ptr() + a, n, n, 0, out.data_ptr(), cap, C.byref(cnt), sp))

    # warm-up of every shape, then the timed pass on a fresh set (records kept for the parity check)
    warm = m.flows(n_flows)
    for c in range(n_calls):
        flows_call(warm, c)
        batch_call(c)
        packed_call(c)
    warm.close()
    fs = m.flows(n_flows)
    got = []
    t_flows, t_batch, t_packed = [], [], []
    for c in range(n_calls):
        t_flows.append(ev_time(torch, stream, lambda: flows_call(fs, c)))
        info = m.last_info()
        t_batch.append(ev_time(torch, stream, lambda: batch_call(c)))
        t_packed.append(ev_time(torch, stream, lambda: packed_call(c)))
    # the records of the timed pass, read back in a second identical pass (the read-back is not timed)
    fs.close()
    fs = m.flows(n_flows)
    for c in range(n_calls):
        flows_call(fs, c, got)
    res = {"flows": n_flows, "calls": n_calls, "bytes_per_call": round(total / n_calls),
           "flows_ms": round(float(np.mean(t_flows)), 4), "batch_ms": round(float(np.mean(t_batch)), 4),
           "packed_ms": round(float(np.mean(t_packed)), 4),
           "flows_over_batch": round(float(np.mean(t_flows) / np.mean(t_batch)), 3),
           "flows_over_packed": round(float(np.mean(t_flows) / np.mean(t_packed)), 3),
           "flows_gbs": round(total / n_calls / float(np.mean(t_flows)) / 1e6, 1),
           "launches_per_call": int(info["launches"]), "h2d_bytes_per_call": int(info["h2d_bytes"])}

    if kind == "large":
        # the pack kernel alone (profiler run of its own) against a bare device-to-device copy of the same bytes
        from torch.profiler import ProfilerActivity, profile
        fs2 = m.flows(n_flows)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for c in range(n_calls):
                flows_call(fs2, c)
            torch.cuda.synchronize()
        fs2.close()
        pack = [e for e in prof.key_averages() if "pfac_flow_pack_kernel" in e.key]
        pack_us = pack[0].device_time_total / pack[0].count if pack else float("nan")
        src = d_text[:per_call]
        dst = torch.empty_like(src)
        with torch.cuda.stream(stream):   # (a same-dtype device tensor copy is one cudaMemcpyAsync)
            for _ in range(3):
                dst.copy_(src)
            copy_ms = float(np.mean([ev_time(torch, stream, lambda: dst.copy_(src)) for _ in range(10)]))
        packed_bytes = per_call + n_flows * (m.tables.max_pat_len - 1)
        res.update({"pack_ms": round(pack_us / 1e3, 4), "d2d_copy_ms": round(copy_ms, 4),
                    "pack_gbs": round(packed_bytes / (pack_us / 1e3) / 1e6, 1),
                    "d2d_copy_gbs": round(per_call / copy_ms / 1e6, 1),
                    "pack_over_copy_rate": round((packed_bytes / pack_us * 1e3) / (per_call / copy_ms), 3)})

    # parity: per flow, the union of its records over the calls == one scan of its concatenated bytes
    gf = np.concatenate([g[0] for g in got])
    gp = np.concatenate([g[1] for g in got])
    gi = np.concatenate([g[2] for g in got])
    order = np.lexsort((lengths[gi], gp, gf))
    gf, gp, gi = gf[order], gp[order], gi[order]
    starts = np.zeros((n_calls, n_flows), dtype=np.int64)
    for c, (a, offs, ids) in enumerate(calls):
        starts[c][ids] = a + offs[:-1].astype(np.int64)
    stream_len = sizes.sum(axis=0)
    if kind == "packets":
        docs = np.concatenate([text[starts[c][f]:starts[c][f] + sizes[c][f]] for f in range(n_flows) for c in range(n_calls)])
        doffs = np.zeros(n_flows + 1, dtype=np.uint64)
        doffs[1:] = np.cumsum(stream_len)
        wfirst, wrec = m.scan_batch(docs, doffs, cap=len(gf) + (1 << 20))
        wf = np.repeat(np.arange(n_flows), np.diff(wfirst.astype(np.int64)))
        wp, wi = wrec["pos"].astype(np.int64), wrec["id"].astype(np.int64)
    else:
        wf, wp, wi = [], [], []
        for f in range(n_flows):
            s = torch.cat([d_text[starts[c][f]:starts[c][f] + sizes[c][f]] for c in range(n_calls)])
            r = m.scan_device(s, cap=len(s) // 64)
            wf.append(np.full(len(r), f))
            wp.append(r["pos"].astype(np.int64))
            wi.append(r["id"].astype(np.int64))
        wf, wp, wi = np.concatenate(wf), np.concatenate(wp), np.concatenate(wi)
    res["records"] = int(len(gf))
    res["parity_union_equals_whole_stream_scan"] = bool(len(gf) == len(wf) and np.array_equal(gf, wf) and
                                                         np.array_equal(gp, wp) and np.array_equal(gi, wi))
    fs.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("flow_bench.py measures on the GPU; none is available")
    import phfpfac_b200 as pf
    from phfpfac_b200._lib import lib
    import pfac_synth as synth
    from bench import WORKLOADS

    name, power = card()
    pk, count, pseed, lo, hi = WORKLOADS["config3"][:5]
    pats = synth.synth_patterns(pk, count, pseed, lo, hi)
    t = pf.Tables.from_bytes(pats, 1, 256)
    lengths = t.pattern_lengths().astype(np.int64)
    m = pf.Matcher(t, device=0)
    res = {"metric": "streaming scan of many flows", "patterns": "config3 (10,000 synthetic Snort-like)",
           "max_pat_len": t.max_pat_len, "gpu": name, "power_limit": power}
    for kind in ("packets", "large"):
        res[kind] = run(kind, m, lengths, pats, torch, pf, lib, synth)
    res["parity"] = all(res[k]["parity_union_equals_whole_stream_scan"] for k in ("packets", "large"))
    m.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
