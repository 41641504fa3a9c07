"""What the device layer (pfac_device.cu) reports about each scan and each context: pfac_ctx_last_scan_info after
every entry point -- device scan, its asynchronous form, batch scan and the host pipeline over several chunks, one
of them overflowing -- and pfac_ctx_derived_info's table_bytes for sets that upload different table buffers."""
import numpy as np
import pytest

import phfpfac_b200 as pf
import pfac_synth as synth
from test_detector_paths_host import long_tail

pytestmark = pytest.mark.gpu

TILE = 8192          # start positions per tile (kTile, pfac_kernel.cuh)
RESULT_BYTES = 16    # struct Result, copied back once per enqueued host chunk
RECORD_BYTES = 8     # struct pfac_match
BG = 10              # '\n' separates the patterns: no pattern contains it

DIRECT_PATS = synth.synth_patterns(1, 300, 11, 3, 24) + b"a\nab\nabc\nGET /\n"   # patterns of <= 3 bytes


def pattern_set(name):
    """-> (pattern file image, PHF width).  mode0: detector with the one-load `step` layout (width >= 256) and the
    pattern directory; mode0_narrow: the same patterns without `step`; mode2: global mode; long: no pattern
    directory and no batch scans (patterns over 513 bytes); direct: the dense-match kernel alone."""
    mode0 = synth.synth_patterns(1, 3000, 3, 4, 64)
    return {
        "mode0": (mode0, 256),
        "mode0_narrow": (mode0, 64),
        "mode2": (synth.synth_patterns(1, 30000, 7, 4, 12), 256),
        "long": (mode0 + long_tail((600, 900), 77), 256),
        "direct": (DIRECT_PATS, 256),
    }[name]


# derived mode and table_bytes of every set on an NVIDIA B200 (the shared-memory budget sizes the images), as the
# layer computed them when table_bytes was summed by hand from the allocation sizes
TABLE_BYTES = {
    "mode0": (0, 1287384),
    "mode0_narrow": (0, 1151192),
    "mode2": (2, 7754808),
    "long": (0, 1136116),
    "direct": (0, 232820),
}


def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def matcher(name, **kw):
    pats, width = pattern_set(name)
    return pf.Matcher(pf.Tables.from_bytes(pats, 1, width), device=0, **kw), pats


def sm_count():
    return torch_cuda().cuda.get_device_properties(0).multi_processor_count


def ceil_div(a, b):
    return (a + b - 1) // b


def launches_of(name):
    return 1 if name == "direct" else 3   # the dense-match kernel alone / detector + dense-match + ordering pass


def check_device_info(m, name, mis, n_starts, extra_launches=0, h2d=0):
    info = m.last_info()
    tiles = ceil_div(mis + n_starts, TILE)
    want = {"launches": launches_of(name) + extra_launches, "tiles": tiles, "ctas": min(tiles, sm_count()),
            "smem_bytes": m.derived_info()["smem_bytes"], "h2d_bytes": h2d, "d2h_bytes": 0, "chunks": 1,
            "flagged_tiles": 0}
    assert info == want, (name, mis, n_starts, info, want)


@pytest.mark.parametrize("name", ["mode0", "mode2", "direct"])
def test_last_info_after_device_scans(name):
    """scan_device (pfac_scan_device_sync), scan_device_raw (pfac_scan_device) and scan_batch
    (pfac_scan_batch_device_sync) at aligned and misaligned inputs: launches, tiles = ceil((mis + n_starts) / 8192),
    ctas = min(tiles, SMs), the detector's shared memory, the offsets upload of a batch, one chunk."""
    torch = torch_cuda()
    m, pats = matcher(name)
    n = 5 * TILE + 777
    text = synth.synth_text(1, 21, n, patterns=pats)
    d = torch.from_numpy(text).cuda()
    assert d.data_ptr() % 16 == 0
    for off, ns in ((0, n), (3, n - 3), (5, n - 5 - 3000)):
        got = m.scan_device(d, n_starts=ns, n_valid=n - off, offset=off)
        assert len(got) > 0
        check_device_info(m, name, off, ns)

    # asynchronous form on a stream of the caller's: same counters, the count lands in device memory
    cap = 1 << 16
    out = torch.empty((cap, 2), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    st = torch.cuda.Stream()
    off, ns = 7, n - 7 - 100
    m.scan_device_raw(d.data_ptr() + off, ns, n - off, 0, out.data_ptr(), cap, cnt.data_ptr(), st.cuda_stream)
    torch.cuda.synchronize()
    check_device_info(m, name, off, ns)
    want = m.scan_device(d, n_starts=ns, n_valid=n - off, offset=off)
    assert int(cnt.item()) == len(want) and np.array_equal(out[:len(want)].cpu().numpy()[:, 0], want["pos"].astype(np.int32))

    # batch scan: the packed scan's counters plus the three kernels of the split pass and the offsets upload
    sizes = [0, 1, 500, 9000, 20000, 3, n - 29504 - 11]
    offs = np.zeros(len(sizes) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum(sizes)
    for off in (0, 11):
        first, rec = m.scan_batch(d, offs, offset=off)
        assert int(first[-1]) == len(rec) > 0
        check_device_info(m, name, off, int(offs[-1]), extra_launches=3, h2d=4 * len(offs))
    m.close()


def host_expect(m, n, chunk, halo, launches, n_records, overflow=()):
    """Counters of one pfac_scan_host call over n bytes (n_starts = n_valid = n): every chunk enqueued once, the
    chunks in `overflow` a second time (their record buffer grown), the Result block back per enqueue, then every
    record."""
    n_chunks = ceil_div(n, chunk)
    enq = list(range(n_chunks)) + list(overflow)
    h2d = tiles = ctas = 0
    for c in enq:
        off = c * chunk
        ns = min(chunk, n - off)
        h2d += min(ns + halo, n - off)
        tiles += ceil_div(ns, TILE)
        ctas = max(ctas, min(ceil_div(ns, TILE), sm_count()))
    return {"launches": launches * len(enq), "tiles": tiles, "ctas": ctas, "smem_bytes": m.derived_info()["smem_bytes"],
            "h2d_bytes": h2d, "d2h_bytes": RESULT_BYTES * len(enq) + RECORD_BYTES * n_records, "chunks": n_chunks,
            "flagged_tiles": 0}


@pytest.mark.parametrize("name", ["mode0", "mode2"])
def test_last_info_after_host_pipeline(name):
    """scan_host over 6 chunks of 16 KiB and a partial one on 2 streams: h2d = chunk lengths plus halo, d2h = 16
    per chunk plus 8 per record, chunks = 7."""
    m, pats = matcher(name, n_streams=2, chunk_bytes=2 * TILE)
    n = 6 * 2 * TILE + 1234
    text = synth.synth_text(1, 22, n, patterns=pats)
    got = m.scan_host(text, cap=n)
    assert len(got) > 0
    halo = m.tables.max_pat_len - 1
    assert m.last_info() == host_expect(m, n, 2 * TILE, halo, launches_of(name), len(got))
    m.close()


def test_last_info_after_host_overflow():
    """One chunk of the host pipeline (a run of 'a', a match at every position) holds more records than its stage's
    buffer: the buffer grows and the chunk is enqueued again, which counts in launches, tiles, h2d and d2h."""
    m, pats = matcher("direct", n_streams=2, chunk_bytes=2 * TILE)
    chunk = 2 * TILE
    text = np.full(4 * chunk + 100, BG, dtype=np.uint8)
    text[chunk:2 * chunk] = ord("a")
    got = m.scan_host(text, cap=len(text) * 4)
    assert len(got) > max(chunk // 8, 4096)   # more than the stage's record buffer holds at first
    halo = m.tables.max_pat_len - 1
    assert m.last_info() == host_expect(m, len(text), chunk, halo, 1, len(got), overflow=(1,))
    # the grown buffer stays: the same call again does not overflow
    got2 = m.scan_host(text, cap=len(text) * 4)
    assert np.array_equal(got, got2)
    assert m.last_info() == host_expect(m, len(text), chunk, halo, 1, len(got))
    m.close()


@pytest.mark.parametrize("name", list(TABLE_BYTES))
def test_table_bytes(name):
    """Device bytes of a context's tables: canonical arrays, detector image, global-mode image, walk cache, and
    where the set has them the `step` layout, the pattern directory and the pattern lengths of batch scans."""
    m, _ = matcher(name)
    di = m.derived_info()
    mode, table_bytes = TABLE_BYTES[name]
    assert (di["mode"], di["table_bytes"]) == (mode, table_bytes), (name, di)
    m.close()
