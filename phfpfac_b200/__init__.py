"""phfpfac_b200 -- B200-native PFAC matcher: thin Python binding over the C ABI.

Host-side mirror of the reference's operator interface for the scan path
(regex_GPU_PHF/main.cc:35-37 and the thread_data block, main.cc:19-32):

    reference                                   here
    ------------------------------------------  ---------------------------------------------
    create_PFAC_table_reorder + FFDM            Tables.from_file / Tables.from_bytes
    thread_data{s0Table,r,HT,val,HTSize,...}    Tables.part(g)  (canonical arrays, bit-compatible)
    GPU_Malloc_Memory(...)                      Matcher(tables, device=...)
    GPU_TraceTable(...)                         Matcher.scan_host(...) / Matcher.scan_device(...)
    (none: many independent documents)          Matcher.scan_batch(...) / Matcher.scan_docs(...)
    (none: streams of many flows, chunk by chunk) Matcher.flows(n) -> Flows.scan(...) / Flows.feed(...)
    GPU_Free_memory(...)                        Matcher.close()
    merge + fprintf loop (main.cc:304-350)      format_records / write_result

All compute happens in phfpfac_b200/_build/libpfac_b200.so (hand-written sm_100a CUDA); this
module only marshals buffers.  PyTorch, when used, only supplies device memory and streams.
"""
import ctypes as C
import weakref

import numpy as np

from ._lib import PFAC_ERR_OUTPUT_FULL, PfacError, check, lib

PFAC_PATTERNS_ESCAPES = 1
PFAC_PATTERNS_CASELESS = 2   # include/pfac_b200.h: ASCII letters match in either case
PFAC_PATTERNS_CASE_RULES = 4   # include/pfac_b200.h: a set with per-pattern case rules (reported, never passed in)

MATCH_DTYPE = np.dtype([("pos", "<u4"), ("id", "<u4")])   # struct pfac_match
FLOW_MATCH_DTYPE = np.dtype([("pos", "<u8"), ("id", "<u4")])   # a match of a flow: absolute stream position

__all__ = ["Tables", "Matcher", "Flows", "Job", "PfacError", "MATCH_DTYPE", "FLOW_MATCH_DTYPE", "format_records", "write_result",
           "write_sidecar", "read_sidecar", "pattern_file_hash", "pinned", "device_count", "plan_shard"]


def _as_u8(data):
    """The caller's bytes as a flat uint8 array WITHOUT a copy where they already are one (pinned buffers keep
    their address); anything that is not made of single bytes is refused rather than reinterpreted."""
    if isinstance(data, np.ndarray):
        if data.dtype.itemsize != 1:
            raise TypeError(f"input must be an array of bytes (uint8), not {data.dtype}")
        return np.ascontiguousarray(data).view(np.uint8).reshape(-1)
    return np.frombuffer(bytes(data), dtype=np.uint8)


def _until_fits(scan, cap):
    """scan(cap) -> (rc, count, buffers), called again with cap = count while the records do not fit
    (PFAC_ERR_OUTPUT_FULL: count is then the capacity they need).  -> (buffers, count) of the call that fit."""
    while True:
        rc, count, bufs = scan(cap)
        if rc != PFAC_ERR_OUTPUT_FULL:
            check(rc)
            return bufs, count
        cap = count


def _records(out, n):
    """The first n records of an int32 [cap, 2] torch device buffer as a MATCH_DTYPE array."""
    rec = out[:n].cpu().numpy().astype(np.uint32).reshape(-1, 2)
    res = np.zeros(n, dtype=MATCH_DTYPE)
    res["pos"], res["id"] = rec[:, 0], rec[:, 1]
    return res


def _arr(ptr, n):
    if n <= 0 or not ptr:
        return np.zeros(0, dtype=np.int32)
    return np.ctypeslib.as_array(ptr, shape=(n,)).copy()


class PartView:
    """Canonical arrays of one partition -- the table half of thread_data (main.cc:19-32)."""

    def __init__(self, t, g):
        info = (C.c_int32 * 9)()
        check(lib.pfac_tables_part_info(t._h, g, info))
        (self.state_num, self.n_final, self.max_len, self.ht_size, self.n_r, self.n_keys, self.max_key,
         self.max_offset, self.min_len) = list(info)
        self.width = t.width
        self.s0 = _arr(lib.pfac_tables_s0(t._h, g), 256)
        self.r = _arr(lib.pfac_tables_r(t._h, g), self.n_r)
        self.HT = _arr(lib.pfac_tables_HT(t._h, g), self.ht_size)
        self.val = _arr(lib.pfac_tables_val(t._h, g), self.ht_size)
        self.idmap = _arr(lib.pfac_tables_idmap(t._h, g), self.n_final)


class Tables:
    """PFAC trie + PHF arrays (create_PFAC_table_reorder.c:6, phf.c:151)."""

    def __init__(self, handle):
        self._h = handle
        self.n_parts = lib.pfac_tables_n_parts(handle)
        self.n_patterns = lib.pfac_tables_n_patterns(handle)
        self.max_pat_len = lib.pfac_tables_max_pat_len(handle)
        self.width = lib.pfac_tables_width(handle)

    @classmethod
    def from_file(cls, path, n_parts=1, width=256, escapes=False, caseless=False):
        h = C.c_void_p()
        rules = _rules(caseless)
        if rules is None:
            check(lib.pfac_tables_build_file_ext(str(path).encode(), n_parts, width, _flags(escapes, caseless), C.byref(h)))
        else:
            check(lib.pfac_tables_build_file_rules(str(path).encode(), n_parts, width, _flags(escapes, False),
                                                   rules.ctypes.data, len(rules), C.byref(h)))
        return cls(h)

    @classmethod
    def from_bytes(cls, data, n_parts=1, width=256, escapes=False, caseless=False):
        """escapes=True: read_pattern_ext / fgetc_ext front-end (create_table_reorder.c:131, ctdef.h:37).
        caseless=True: ASCII letters match in either case (PFAC_PATTERNS_CASELESS): the patterns are folded to
        lower case after the reader, and every scan with these tables folds its text on the device first.
        caseless=[bool per pattern]: per-pattern case rules (one per pattern the reader returns): True matches in
        either case, False byte for byte.  Uniform rules give exactly the caseless=True / False set."""
        data = bytes(data)
        h = C.c_void_p()
        rules = _rules(caseless)
        if rules is None:
            check(lib.pfac_tables_build_mem_ext(data, len(data), n_parts, width, _flags(escapes, caseless), C.byref(h)))
        else:
            check(lib.pfac_tables_build_mem_rules(data, len(data), n_parts, width, _flags(escapes, False),
                                                  rules.ctypes.data, len(rules), C.byref(h)))
        return cls(h)

    @classmethod
    def from_arrays(cls, s0, r, HT, val, width, state_num, n_final, idmap, max_pat_len):
        a = [np.ascontiguousarray(x, dtype=np.int32) for x in (s0, r, HT, val, idmap)]
        h = C.c_void_p()
        check(lib.pfac_tables_from_arrays(a[0].ctypes.data, a[1].ctypes.data, len(a[1]), a[2].ctypes.data,
                                          a[3].ctypes.data, len(a[2]), width, state_num, n_final,
                                          a[4].ctypes.data, max_pat_len, C.byref(h)))
        return cls(h)

    @classmethod
    def load(cls, path):
        """A table set saved with save() (checksummed cache of the canonical arrays)."""
        h = C.c_void_p()
        check(lib.pfac_tables_load(str(path).encode(), C.byref(h)))
        return cls(h)

    def save(self, path):
        check(lib.pfac_tables_save(self._h, str(path).encode()))

    @property
    def caseless(self):
        """True for a set built with caseless=True or all rules True (also after save / load); False for mixed rules."""
        return bool(lib.pfac_tables_flags(self._h) & PFAC_PATTERNS_CASELESS)

    @property
    def case_rules(self):
        """np.uint8[n_patterns]: 1 where pattern id i + 1 matches in either case, 0 where it matches byte for byte."""
        out = np.zeros(self.n_patterns, dtype=np.uint8)
        if self.n_patterns:
            check(lib.pfac_tables_case_rules(self._h, out.ctypes.data, len(out)))
        return out

    def source_hash(self):
        """Hash of the pattern file image + reader flags the set was built from (0: wrapped from arrays)."""
        return int(lib.pfac_tables_source_hash(self._h))

    def part(self, g=0):
        return PartView(self, g)

    def derive_check(self, g=0, t2_bytes=32768, t3_bytes=32768, tm2_bytes=32768):
        """Host-side build + verification of the detector's shared-memory filters (no GPU needed)."""
        st = (C.c_uint64 * 10)()
        check(lib.pfac_tables_derive_check(self._h, g, t2_bytes, t3_bytes, tm2_bytes, st))
        keys = ("image_bytes", "t1_pairs", "t2_set", "prefixes4", "has_short", "has_t3", "tm_keys", "tm2_keys",
                "t3_set", "tm2_bits")
        return dict(zip(keys, list(st)))

    def filter_profile(self, text, g=0, t2_bytes=32768, t3_bytes=32768, tm2_bytes=32768):
        """Diagnostics: survivors per stage of the detector's filter cascade over `text` (host model, counts only)."""
        buf = np.ascontiguousarray(text, dtype=np.uint8)
        c = (C.c_uint64 * 12)()
        check(lib.pfac_tables_filter_profile(self._h, g, t2_bytes, t3_bytes, tm2_bytes, buf.ctypes.data, len(buf), c))
        keys = ("positions", "t1_pass", "prefix_found", "window1_pass", "window2_pass", "bypass", "to_emit",
                "slices_flagged", "slices")
        return dict(zip(keys, list(c)))

    def pattern_lengths(self, g=0):
        """np.int32[n_ids]: the length of every pattern id of partition g (0 for ids no final state reports:
        the earlier copies of a duplicated line).  Refused (PfacError) for automata that are not trees."""
        n = C.c_int32(0)
        check(lib.pfac_tables_pattern_lengths(self._h, g, None, 0, C.byref(n)))
        out = np.zeros(n.value, dtype=np.int32)
        if n.value:
            check(lib.pfac_tables_pattern_lengths(self._h, g, out.ctypes.data, n.value, C.byref(n)))
        return out

    def lookup(self, state, byte, g=0):
        return lib.pfac_tables_lookup(self._h, g, state, byte)

    def close(self):
        if self._h and lib is not None:
            lib.pfac_tables_destroy(self._h)
        self._h = None

    def __del__(self):
        self.close()


def _rules(caseless):
    """None for one rule for the whole set (a bool), else the per-pattern rules as a uint8 array."""
    if np.ndim(caseless) == 0:
        return None
    return np.ascontiguousarray([1 if c else 0 for c in caseless], dtype=np.uint8)


def _flags(escapes, caseless):
    return (PFAC_PATTERNS_ESCAPES if escapes else 0) | (PFAC_PATTERNS_CASELESS if caseless else 0)


def pattern_file_hash(path, escapes=False, caseless=False):
    """The source hash of the set from_file(path, escapes=..., caseless=...) builds (caseless: a bool or one per pattern)."""
    h = C.c_uint64(0)
    rules = _rules(caseless)
    if rules is None:
        check(lib.pfac_pattern_file_hash(str(path).encode(), _flags(escapes, caseless), C.byref(h)))
    else:
        check(lib.pfac_pattern_file_hash_rules(str(path).encode(), _flags(escapes, False), rules.ctypes.data, len(rules),
                                               C.byref(h)))
    return h.value


def device_count():
    n = C.c_int(0)
    check(lib.pfac_device_count(C.byref(n)))
    return n.value


class Matcher:
    """One device: tables uploaded once, then scans (GPU_Malloc_Memory/GPU_TraceTable/GPU_Free_memory)."""

    def __init__(self, tables, device=0, part=0, n_streams=4, chunk_bytes=0):
        self._h = None
        h = C.c_void_p()
        check(lib.pfac_ctx_create(device, tables._h, part, n_streams, chunk_bytes, C.byref(h)))
        self._h = h
        self.tables = tables
        self.device = device
        self._flows = weakref.WeakSet()

    def close(self):
        for f in list(getattr(self, "_flows", ())):   # a flow set must not outlive its context
            f.close()
        if self._h and lib is not None:
            lib.pfac_ctx_destroy(self._h)
        self._h = None

    def flows(self, n_flows):
        """A set of n_flows independent streams scanned chunk by chunk (Flows)."""
        f = Flows(self, n_flows)
        self._flows.add(f)
        return f

    def __del__(self):
        self.close()

    def last_info(self):
        info = (C.c_uint64 * 8)()
        check(lib.pfac_ctx_last_scan_info(self._h, info))
        keys = ("launches", "tiles", "ctas", "smem_bytes", "h2d_bytes", "d2h_bytes", "chunks", "flagged_tiles")
        return dict(zip(keys, list(info)))

    def set_timing(self, enable=True):
        check(lib.pfac_ctx_set_timing(self._h, 1 if enable else 0))

    def kernel_time(self):
        """(total ms, launches) of the detector kernel since the last call (needs set_timing)."""
        ms, n = C.c_double(0), C.c_int(0)
        check(lib.pfac_ctx_kernel_time(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def derived_info(self):
        info = (C.c_uint64 * 16)()
        check(lib.pfac_ctx_derived_info(self._h, info))
        keys = ("image_bytes", "t1_pairs", "t2_bits", "t2_set", "prefixes4", "has_short", "tm_keys", "tm2_keys",
                "t3_bits", "t3_set", "smem_bytes", "table_bytes", "ring_stages", "tm2_bits", "mode", "tm_bits")
        return dict(zip(keys, list(info)))

    # -- device-resident input (raw pointers; torch tensors are accepted for convenience)
    def scan_device_raw(self, d_in, n_starts, n_valid, base_pos, d_out, cap, d_count, stream=0):
        check(lib.pfac_scan_device(self._h, d_in, n_starts, n_valid, base_pos, d_out, cap, d_count, stream))

    def scan_device(self, t_in, n_starts=None, n_valid=None, base_pos=0, cap=None, offset=0):
        """t_in: torch uint8 CUDA tensor.  Returns a MATCH_DTYPE array (synchronous)."""
        import torch
        total = t_in.numel() - offset
        n_valid = total if n_valid is None else n_valid
        n_starts = n_valid if n_starts is None else n_starts
        cap = max(1024, n_starts // 8) if cap is None else cap

        def scan(cap):
            out = torch.empty((max(cap, 1), 2), dtype=torch.int32, device=t_in.device)
            cnt = C.c_uint64(0)
            # on torch's current stream: ordered after whatever produced t_in (and allocated `out`) there
            stream = torch.cuda.current_stream(t_in.device).cuda_stream
            if stream == 0:     # the legacy default stream: 0 means "the library's own stream" to the C ABI
                torch.cuda.current_stream(t_in.device).synchronize()
            rc = lib.pfac_scan_device_sync(self._h, t_in.data_ptr() + offset, n_starts, n_valid, base_pos,
                                           out.data_ptr(), cap, C.byref(cnt), stream or None)
            return rc, cnt.value, out

        out, n = _until_fits(scan, cap)
        return _records(out, n)

    # -- many independent documents packed back to back: one launch sequence, per-document results
    def scan_batch(self, values, offsets, cap=None, offset=0):
        """values: torch uint8 CUDA tensor (or host bytes / uint8 array, uploaded through torch) holding the
        documents back to back from byte `offset` on; offsets: n_docs + 1 integers, document i = bytes
        [offsets[i], offsets[i+1]).  Returns (doc_first: np.uint64[n_docs + 1], records: MATCH_DTYPE): the records
        of document i are records[doc_first[i]:doc_first[i+1]], positions relative to the document -- exactly
        what scan_device returns for that document alone (synchronous)."""
        import torch
        if not isinstance(values, torch.Tensor):
            values = torch.from_numpy(_as_u8(values).copy()).cuda(self.device)
        offs = np.asarray(offsets)
        if offs.ndim != 1 or len(offs) < 1 or not np.issubdtype(offs.dtype, np.integer):
            raise ValueError("offsets must be a 1-D sequence of n_docs + 1 integers")
        if (offs < 0).any() or int(offs.max()) > values.numel() - offset:
            raise ValueError("offsets point outside the values")
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        n_docs = len(offs) - 1
        cap = max(1024, int(offs[-1]) // 8) if cap is None else cap
        stream = torch.cuda.current_stream(values.device).cuda_stream

        def scan(cap):
            out = torch.empty((max(cap, 1), 2), dtype=torch.int32, device=values.device)
            first = torch.empty(n_docs + 1, dtype=torch.int64, device=values.device)
            cnt = C.c_uint64(0)
            if stream == 0:     # the legacy default stream: 0 means "the library's own stream" to the C ABI
                torch.cuda.current_stream(values.device).synchronize()
            rc = lib.pfac_scan_batch_device_sync(self._h, values.data_ptr() + offset if values.numel() else None,
                                                 offs.ctypes.data, n_docs, out.data_ptr(), cap, first.data_ptr(),
                                                 C.byref(cnt), stream or None)
            return rc, cnt.value, (out, first)

        (out, first), n = _until_fits(scan, cap)
        return first.cpu().numpy().view(np.uint64), _records(out, n)

    def scan_docs(self, docs):
        """docs: list of bytes-like documents -> list of per-document MATCH_DTYPE arrays (one batch scan)."""
        parts = [_as_u8(d) for d in docs]
        offs = np.zeros(len(parts) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(p) for p in parts], dtype=np.uint64)
        buf = np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint8)
        first, rec = self.scan_batch(buf, offs)
        return [rec[int(first[i]):int(first[i + 1])] for i in range(len(parts))]

    # -- host input: H2D + kernel + D2H pipeline
    def scan_host(self, data, n_starts=None, base_pos=0, cap=None):
        buf = _as_u8(data)
        n_valid = len(buf)
        n_starts = n_valid if n_starts is None else n_starts
        cap = max(1024, n_starts // 8) if cap is None else cap

        def scan(cap):
            out = np.zeros(max(cap, 1), dtype=MATCH_DTYPE)
            cnt = C.c_uint64(0)
            rc = lib.pfac_scan_host(self._h, buf.ctypes.data if len(buf) else None, n_starts, n_valid, base_pos,
                                    out.ctypes.data, cap, C.byref(cnt))
            return rc, cnt.value, out

        out, n = _until_fits(scan, cap)
        return out[:n]


class Flows:
    """Streams of many flows (pfac_flows_*, pfac_scan_flows_device_sync): each call scans one chunk for each of
    several distinct flows and reports the matches that END in the chunk, straddling chunk boundaries included,
    so the union of a flow's records equals one scan of its whole stream.  A call that fails (records beyond cap,
    bad arguments) leaves every flow unchanged.  Keeps its Matcher alive; Matcher.close() closes it first."""

    def __init__(self, matcher, n_flows):
        self._h = None
        h = C.c_void_p()
        check(lib.pfac_flows_create(matcher._h, n_flows, C.byref(h)))
        self._h = h
        self.matcher = matcher
        self.n_flows = n_flows

    def close(self):
        if self._h and lib is not None:
            lib.pfac_flows_destroy(self._h)
        self._h = None

    def __del__(self):
        self.close()

    def reset(self, flow):
        """flow starts a new stream: position 0, nothing carried."""
        check(lib.pfac_flows_reset(self._h, flow))

    def position(self, flow):
        """Bytes flow has consumed so far."""
        n = C.c_uint64(0)
        check(lib.pfac_flows_position(self._h, flow, C.byref(n)))
        return n.value

    def scan(self, flow_ids, values, offsets, cap=None, offset=0):
        """values: torch uint8 CUDA tensor (or host bytes / uint8 array, uploaded through torch) holding the chunks
        back to back from byte `offset` on; offsets: n + 1 integers, chunk i = bytes [offsets[i], offsets[i+1]), for
        flow flow_ids[i] (distinct).  Returns (chunk_first: np.uint64[n + 1], base: np.uint64[n], records:
        MATCH_DTYPE): the records of chunk i are records[chunk_first[i]:chunk_first[i+1]], ordered by (pos, pattern
        length), at stream positions base[i] + pos (synchronous)."""
        import torch
        m = self.matcher
        if not isinstance(values, torch.Tensor):
            values = torch.from_numpy(_as_u8(values).copy()).cuda(m.device)
        offs = np.asarray(offsets)
        if offs.ndim != 1 or len(offs) < 1 or not np.issubdtype(offs.dtype, np.integer):
            raise ValueError("offsets must be a 1-D sequence of n + 1 integers")
        if (offs < 0).any() or int(offs.max()) > values.numel() - offset:
            raise ValueError("offsets point outside the values")
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        ids = np.ascontiguousarray(flow_ids, dtype=np.uint32).reshape(-1)
        n = len(offs) - 1
        if len(ids) != n:
            raise ValueError("one flow id per chunk")
        carried = n * max(m.tables.max_pat_len - 1, 0)
        cap = max(1024, (int(offs[-1]) + carried) // 8) if cap is None else cap
        base = np.zeros(n, dtype=np.uint64)
        stream = torch.cuda.current_stream(values.device).cuda_stream

        def scan(cap):
            out = torch.empty((max(cap, 1), 2), dtype=torch.int32, device=values.device)
            first = torch.empty(n + 1, dtype=torch.int64, device=values.device)
            cnt = C.c_uint64(0)
            if stream == 0:     # the legacy default stream: 0 means "the library's own stream" to the C ABI
                torch.cuda.current_stream(values.device).synchronize()
            rc = lib.pfac_scan_flows_device_sync(self._h, values.data_ptr() + offset if values.numel() else None,
                                                 offs.ctypes.data, ids.ctypes.data, n, out.data_ptr(), cap,
                                                 first.data_ptr(), base.ctypes.data, C.byref(cnt), stream or None)
            return rc, cnt.value, (out, first)

        (out, first), count = _until_fits(scan, cap)   # (exact: a call that does not fit commits nothing)
        return first.cpu().numpy().view(np.uint64), base, _records(out, count)

    def feed(self, flow_ids, chunks):
        """chunks: bytes-like chunks for the distinct flows flow_ids -> one FLOW_MATCH_DTYPE array per chunk, with
        absolute stream positions (one call)."""
        parts = [_as_u8(c) for c in chunks]
        offs = np.zeros(len(parts) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(p) for p in parts], dtype=np.uint64)
        buf = np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint8)
        first, base, rec = self.scan(flow_ids, buf, offs)
        res = []
        for i in range(len(parts)):
            seg = rec[int(first[i]):int(first[i + 1])]
            r = np.zeros(len(seg), dtype=FLOW_MATCH_DTYPE)
            r["pos"] = seg["pos"].astype(np.uint64) + base[i]
            r["id"] = seg["id"]
            res.append(r)
        return res


class Job:
    """All GPUs of the box: input sharded in contiguous chunks (+halo) -- the loop of main.cc:171-272."""

    def __init__(self, tables, devices=None, streams_per_gpu=4, chunk_bytes=0):
        self._h = None
        if devices is None:
            devices = list(range(device_count()))
        arr = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        check(lib.pfac_job_create(tables._h, arr, len(devices), streams_per_gpu, chunk_bytes, C.byref(h)))
        self._h = h
        self.tables = tables

    def run(self, data):
        """-> (total matches, [(base position, uint32 array [count, 2] of (pos - base, id)), ...] in position order)."""
        buf = _as_u8(data)
        n = C.c_uint64(0)
        check(lib.pfac_job_run(self._h, buf.ctypes.data if len(buf) else None, len(buf), C.byref(n)))
        return n.value, self._segments()

    def _segments(self):
        segs = []
        for i in range(lib.pfac_job_n_segments(self._h)):
            base, cnt, ptr = C.c_uint64(0), C.c_uint64(0), C.c_void_p()
            check(lib.pfac_job_segment(self._h, i, C.byref(base), C.byref(ptr), C.byref(cnt)))
            if cnt.value:
                a = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint32)), shape=(cnt.value, 2)).copy()
            else:
                a = np.zeros((0, 2), dtype=np.uint32)
            segs.append((base.value, a))
        return segs

    def run_file(self, path, n):
        """pfac_job_run_file: scan the first n bytes of a file, read chunk by chunk while scanning."""
        nm = C.c_uint64(0)
        check(lib.pfac_job_run_file(self._h, str(path).encode(), n, C.byref(nm)))
        return nm.value, self._segments()

    def close(self):
        if self._h and lib is not None:
            lib.pfac_job_destroy(self._h)
        self._h = None

    def __del__(self):
        self.close()


class pinned:
    """Context manager: pin a numpy array in place (pfac_host_register) for link-speed H2D copies."""

    def __init__(self, arr, read_only=False):
        self.arr, self.read_only, self.ok = arr, read_only, False

    def __enter__(self):
        check(lib.pfac_host_register(self.arr.ctypes.data, self.arr.nbytes, int(self.read_only)))
        self.ok = True
        return self.arr

    def __exit__(self, *exc):
        if self.ok:
            lib.pfac_host_unregister(self.arr.ctypes.data)
        return False


def plan_shard(n, n_shards, max_pat_len, i):
    """pfac_job_plan: (start, n_starts, n_valid) of shard i -- contiguous chunk + halo of max_pat_len-1."""
    a, b, c = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    check(lib.pfac_job_plan(n, n_shards, max_pat_len, i, C.byref(a), C.byref(b), C.byref(c)))
    return a.value, b.value, c.value


def format_records(records, base_pos=0):
    """main.cc:344 line format for a MATCH_DTYPE array -> bytes."""
    rec = np.ascontiguousarray(records, dtype=MATCH_DTYPE)
    need = lib.pfac_format_records(base_pos, rec.ctypes.data if len(rec) else None, len(rec), None, 0)
    buf = C.create_string_buffer(need + 1)
    lib.pfac_format_records(base_pos, rec.ctypes.data if len(rec) else None, len(rec), buf, need)
    return buf.raw[:need]


def write_result(path, segments):
    """segments: iterable of (base_pos, MATCH_DTYPE array).  Writes GPU_match_result.txt (main.cc:335-350)."""
    w = C.c_void_p()
    check(lib.pfac_write_begin(str(path).encode(), C.byref(w)))
    try:
        for base, rec in segments:
            rec = np.ascontiguousarray(rec, dtype=MATCH_DTYPE)
            check(lib.pfac_write_records(w, base, rec.ctypes.data if len(rec) else None, len(rec)))
    finally:
        check(lib.pfac_write_end(w))


def write_sidecar(path, segments):
    """segments: iterable of (base_pos, MATCH_DTYPE array).  Writes the binary sidecar of the compact records
    (include/pfac_b200.h, pfac_sidecar_*): 8 bytes per match; the text file is a pure function of it."""
    w = C.c_void_p()
    check(lib.pfac_sidecar_begin(str(path).encode(), C.byref(w)))
    try:
        for base, rec in segments:
            rec = np.ascontiguousarray(rec, dtype=MATCH_DTYPE)
            check(lib.pfac_sidecar_records(w, base, rec.ctypes.data if len(rec) else None, len(rec)))
    finally:
        check(lib.pfac_sidecar_end(w))


def read_sidecar(path):
    """-> (pos: uint64 absolute start positions, id: uint32 pattern ids) in file (= position) order."""
    n = C.c_uint64(0)
    check(lib.pfac_sidecar_read(str(path).encode(), None, None, 0, C.byref(n)))
    pos = np.empty(n.value, dtype=np.uint64)
    ids = np.empty(n.value, dtype=np.uint32)
    check(lib.pfac_sidecar_read(str(path).encode(), pos.ctypes.data, ids.ctypes.data, n.value, C.byref(n)))
    return pos, ids
