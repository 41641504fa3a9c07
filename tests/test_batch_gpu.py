"""Batch scan of independent documents (pfac_scan_batch_device / Matcher.scan_batch): every document's records
equal what the oracle -- and pfac_scan_device -- return for that document alone."""
import ctypes as C

import numpy as np
import pytest

import phfpfac_b200 as pf
import pfac_synth as synth
from _oracle import Oracle
from phfpfac_b200._lib import PFAC_ERR_ARG, PFAC_ERR_LIMIT, PFAC_ERR_OUTPUT_FULL, lib

pytestmark = pytest.mark.gpu


def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def pack(docs):
    parts = [np.frombuffer(bytes(d), dtype=np.uint8) if not isinstance(d, np.ndarray) else d for d in docs]
    offs = np.zeros(len(parts) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(p) for p in parts])
    return (np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint8)), offs, parts


class DeviceOracle:
    """pfac_scan_device of one document alone (the batch semantics' definition), for sets too large for the
    oracle's quadratic table build."""

    def __init__(self, m):
        self.m = m

    def scan(self, doc):
        torch = torch_cuda()
        d = torch.from_numpy(np.array(doc, dtype=np.uint8)).cuda() if len(doc) else torch.zeros(16, dtype=torch.uint8, device="cuda")
        got = self.m.scan_device(d, n_starts=len(doc), n_valid=len(doc))
        return got["pos"].astype(np.int64), got["id"].astype(np.int32)


def check_batch(m, oracle, docs, offset=0, cap=None):
    """scan_batch of `docs` (from byte `offset` of the device buffer) == the oracle per document."""
    torch = torch_cuda()
    buf, offs, parts = pack(docs)
    d = torch.zeros(offset + len(buf) + 16, dtype=torch.uint8, device="cuda")
    if len(buf):
        d[offset:offset + len(buf)] = torch.from_numpy(buf.copy()).cuda()
    first, rec = m.scan_batch(d, offs, cap=cap, offset=offset)
    info = m.last_info()
    assert first.dtype == np.uint64 and len(first) == len(parts) + 1
    k = 0
    for i, p in enumerate(parts):
        pos, ids = oracle.scan(p)
        assert int(first[i]) == k, i
        seg = rec[int(first[i]):int(first[i + 1])]
        assert len(seg) == len(pos), (i, len(seg), len(pos))
        assert np.array_equal(seg["pos"].astype(np.int64), pos) and np.array_equal(seg["id"].astype(np.int32), ids), i
        k += len(pos)
    assert int(first[-1]) == k == len(rec)
    return first, rec, info


def random_sizes(rng, n, lo, hi):
    return [int(x) for x in rng.integers(lo, hi, n)]


def cut(text, sizes, rng=None):
    docs, at = [], 0
    for s in sizes:
        if at + s > len(text):
            at = 0
        docs.append(text[at:at + s])
        at += s
    return docs


@pytest.mark.parametrize("seed", range(10))
def test_random_batches(seed):
    """Alphabets and lengths of test_random_patterns_and_texts; documents of 0, 1, shorter than the shortest
    pattern, tile-edge sizes, several tiles and random sizes."""
    rng = np.random.default_rng(1000 + seed)
    alpha = [2, 3, 4, 8, 26, 64, 200, 256, 5, 2][seed]
    n_pat = int(rng.integers(1, 2000))
    max_len = int(rng.integers(1, [6, 12, 40, 100, 20, 64, 16, 30, 300, 700][seed]))
    max_len = min(max_len, 513)   # longer patterns: batches are refused (test_refusals)
    pats = set()
    usable = alpha - (1 if alpha > 10 else 0)
    possible = sum(usable ** L for L in range(1, min(max_len, 8) + 1))
    for _ in range(50 * n_pat):
        if len(pats) >= min(n_pat, possible):
            break
        L = int(rng.integers(1, max_len + 1))
        p = bytes(rng.integers(0, alpha, L).astype(np.uint8))
        if b"\n" not in p:
            pats.add(p)
    blob = b"".join(p + b"\n" for p in pats)
    shortest = min(len(p) for p in pats)
    text = rng.integers(0, alpha, 300000).astype(np.uint8)
    sizes = [0, 1, max(shortest - 1, 0), 0, 8191, 8192, 8193, 16383, 16384, 16385, 3 * 16384 + 77, 0, 0]
    sizes += random_sizes(rng, 40, 0, 3000)
    rng.shuffle(sizes)
    t = pf.Tables.from_bytes(blob, 1, int(2 ** rng.integers(4, 13)))
    m = pf.Matcher(t, device=0)
    check_batch(m, Oracle(blob, 1, 256), cut(text, sizes))
    m.close()


def test_straddling_matches():
    pats = b"needle\nle\nhaystack\nkhay\nk\n"
    o = Oracle(pats, 1, 256)
    m = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256), device=0)
    docs = [b"xxnee", b"dlexx", b"", b"", b"", b"stack needle", b"needle", b"hay", b"", b"stack", b"k", b"hay"]
    first, rec, _ = check_batch(m, o, docs)
    # "nee|dle" across documents 0/1 is absent, "needle" ending exactly at the end of document 6 is present
    assert first[1] - first[0] == 0
    d6 = rec[int(first[6]):int(first[7])]
    assert (d6["pos"] == 0).any() and len(d6) == 2       # needle + le
    # the packed buffer alone does report the straddling matches
    buf, offs, _ = pack(docs)
    pos, _ = o.scan(buf)
    assert len(pos) > len(rec)
    m.close()


def test_kernel_paths(fixtures):
    """DIRECT dense-first set, mode-0 set, global-mode set, a set without a pattern directory."""
    rng = np.random.default_rng(3)
    one_m = np.frombuffer(fixtures["1M"], dtype=np.uint8)
    p3 = synth.synth_patterns(1, 10000, 3, 4, 64)
    p4 = synth.synth_patterns(0, 100000, 5, 8, 32)
    long1 = bytes(rng.integers(97, 100, 300).astype(np.uint8))
    p5 = long1 + b"\n" + long1[:70] + b"\nabcab\nab\nb\n"
    t5 = bytearray(rng.integers(97, 100, 400000).astype(np.uint8).tobytes())
    for s in range(0, 400000 - 300, 9000):
        t5[s:s + 300] = long1
    cases = [  # pattern set, text, what the context must be, oracle
        (fixtures["dictionary"], one_m, lambda i: i["has_short"] == 1, lambda: Oracle(fixtures["dictionary"], 4, 256)),
        (p3, synth.synth_text(1, 4, 4 << 20, patterns=p3), lambda i: i["mode"] == 0, lambda: Oracle(p3, 8, 4096)),
        (p4, synth.synth_text(0, 6, 4 << 20, patterns=p4), lambda i: i["mode"] == 2, None),
        (p5, np.frombuffer(bytes(t5), dtype=np.uint8), lambda i: True, lambda: Oracle(p5, 1, 256)),
    ]
    for pats, text, shape, oracle in cases:
        m = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256), device=0)
        assert shape(m.derived_info())
        sizes = random_sizes(rng, 120 if oracle else 40, 0, 40000) + [0, 16384, 1, 0, 100000]
        info = check_batch(m, oracle() if oracle else DeviceOracle(m), cut(text, sizes))[2]
        assert info["launches"] >= 4         # the packed scan (1 or 3 launches) + the split pass (3)
        m.close()


def test_one_document_equals_scan_device(fixtures):
    torch = torch_cuda()
    pats = fixtures["xab"]
    m = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256), device=0)
    data = np.frombuffer(fixtures["1M"][:700001], dtype=np.uint8)
    d = torch.from_numpy(data.copy()).cuda()
    want = m.scan_device(d)
    first, rec = m.scan_batch(d, [0, len(data)])
    assert first.tolist() == [0, len(want)] and np.array_equal(rec, want)
    assert len(m.scan_docs([data])[0]) == len(want)
    m.close()


def test_alternating_with_scan_device_and_streams(fixtures):
    torch = torch_cuda()
    pats = fixtures["xac"]
    o = Oracle(pats, 1, 256)
    m = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256), device=0)
    rng = np.random.default_rng(11)
    base = np.frombuffer(fixtures["1M"], dtype=np.uint8)
    docs = cut(base, random_sizes(rng, 300, 0, 3000))
    whole = base[:500000].copy()
    want_whole = o.scan(whole)
    d_whole = torch.from_numpy(whole).cuda()
    streams = [torch.cuda.current_stream(), torch.cuda.Stream(), torch.cuda.Stream()]
    for rep in range(6):
        with torch.cuda.stream(streams[rep % 3]):
            check_batch(m, o, docs)
            got = m.scan_device(d_whole)
            assert np.array_equal(got["pos"].astype(np.int64), want_whole[0]) and np.array_equal(got["id"].astype(np.int32), want_whole[1])
    # async calls on two streams without a host sync between them: the context orders them on the device
    buf, offs, parts = pack(docs)
    d = torch.from_numpy(buf.copy()).cuda()
    first_all, rec_all = m.scan_batch(d, offs)
    cap = len(rec_all) + 16
    outs = [torch.full((cap, 2), -1, dtype=torch.int32, device="cuda") for _ in range(2)]
    firsts = [torch.full((len(parts) + 1,), -1, dtype=torch.int64, device="cuda") for _ in range(2)]
    cnts = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(2)]
    offs2 = np.ascontiguousarray(offs[:101])   # the first 100 documents
    torch.cuda.synchronize()
    for rep in range(4):
        i = rep & 1
        o_ = offs if i == 0 else offs2
        assert lib.pfac_scan_batch_device(m._h, d.data_ptr(), o_.ctypes.data, len(o_) - 1, outs[i].data_ptr(), cap,
                                          firsts[i].data_ptr(), cnts[i].data_ptr(), streams[1 + i].cuda_stream) == 0
    torch.cuda.synchronize()
    for i, o_ in enumerate((offs, offs2)):
        n = int(cnts[i].item())
        fr = firsts[i][:len(o_)].cpu().numpy()
        assert n == int(fr[-1]) == int(first_all[len(o_) - 1])
        assert np.array_equal(fr, first_all[:len(o_)].astype(np.int64))
        got = outs[i][:n].cpu().numpy().astype(np.uint32)
        assert np.array_equal(got[:, 0], rec_all["pos"][:n]) and np.array_equal(got[:, 1], rec_all["id"][:n])
    m.close()


def test_misaligned_input():
    pats = b"abcab\nab\nb\ncabcabcabc\nabcabcabcabcabcabcabcabcabcabcabcab\n"
    o = Oracle(pats, 1, 256)
    m = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256), device=0)
    base = np.frombuffer((b"abc" * 30000)[:70001], dtype=np.uint8)
    rng = np.random.default_rng(2)
    docs = cut(base, random_sizes(rng, 30, 0, 2000) + [17000, 5])
    for off in range(0, 18):
        check_batch(m, o, docs, offset=off)
    m.close()


def test_capacity_and_sentinel():
    """cap below the raw count: OUTPUT_FULL with a count that suffices; nothing written past cap."""
    torch = torch_cuda()
    pats = b"a\naa\naaa\nb\n"
    o = Oracle(pats, 1, 256)
    m = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256), device=0)
    docs = [b"aaaa" * 3000 + b"b", b"a", b"", b"ab" * 5000, b"aaa"] * 3
    buf, offs, parts = pack(docs)
    want = sum(len(o.scan(p)[0]) for p in parts)
    raw = len(o.scan(buf)[0])
    assert raw > want
    d = torch.from_numpy(buf.copy()).cuda()
    for cap in (0, 1, 4095, 5000, want - 1):
        out = torch.full((cap + 4096, 2), 0x5a5a5a5a, dtype=torch.int32, device="cuda")
        first = torch.zeros(len(parts) + 1, dtype=torch.int64, device="cuda")
        cnt = C.c_uint64(0)
        rc = lib.pfac_scan_batch_device_sync(m._h, d.data_ptr(), offs.ctypes.data, len(parts), out.data_ptr(), cap,
                                             first.data_ptr(), C.byref(cnt), None)
        assert rc == PFAC_ERR_OUTPUT_FULL and want <= cnt.value <= raw, (cap, cnt.value)
        assert (out[cap:] == 0x5a5a5a5a).all().item(), cap
        # the rescan with the reported count is exact
        first2, rec = m.scan_batch(d, offs, cap=cnt.value)
        assert len(rec) == want
    check_batch(m, o, docs, cap=1)
    check_batch(m, o, docs, cap=want)
    m.close()


def test_async_form_on_a_torch_stream(fixtures):
    torch = torch_cuda()
    pats = fixtures["xab"]
    m = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256), device=0)
    rng = np.random.default_rng(4)
    docs = cut(np.frombuffer(fixtures["1M"], dtype=np.uint8), random_sizes(rng, 500, 0, 1500))
    first_want, rec_want = m.scan_batch(pack(docs)[0], pack(docs)[1])
    buf, offs, parts = pack(docs)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d = torch.from_numpy(buf.copy()).cuda()
        out = torch.empty((len(rec_want) + 8, 2), dtype=torch.int32, device="cuda")
        first = torch.full((len(parts) + 1,), -1, dtype=torch.int64, device="cuda")
        cnt = torch.full((1,), -1, dtype=torch.int64, device="cuda")
        assert lib.pfac_scan_batch_device(m._h, d.data_ptr(), offs.ctypes.data, len(parts), out.data_ptr(), out.shape[0],
                                          first.data_ptr(), cnt.data_ptr(), s.cuda_stream) == 0
        info = m.last_info()
    s.synchronize()
    assert int(cnt.item()) == len(rec_want)
    assert np.array_equal(first.cpu().numpy().view(np.uint64), first_want)
    got = out[:len(rec_want)].cpu().numpy().astype(np.uint32)
    assert np.array_equal(got[:, 0], rec_want["pos"]) and np.array_equal(got[:, 1], rec_want["id"])
    assert info["launches"] >= 4 and info["h2d_bytes"] == 4 * (len(parts) + 1)


def test_empty_batches():
    torch = torch_cuda()
    m = pf.Matcher(pf.Tables.from_bytes(b"ab\n", 1, 256), device=0)
    d = torch.zeros(16, dtype=torch.uint8, device="cuda")
    first, rec = m.scan_batch(d, [0])
    assert first.tolist() == [0] and len(rec) == 0
    first, rec = m.scan_batch(d, [0, 0, 0, 0])
    assert first.tolist() == [0, 0, 0, 0] and len(rec) == 0
    assert m.scan_docs([]) == [] and [len(x) for x in m.scan_docs([b"", b"ab", b""])] == [0, 1, 0]
    m.close()


def test_refusals(fixtures):
    torch = torch_cuda()
    rng = np.random.default_rng(5)
    d = torch.from_numpy(np.frombuffer(b"abcab" * 100, dtype=np.uint8).copy()).cuda()
    # patterns longer than 513 bytes
    long1 = bytes(rng.integers(97, 100, 514).astype(np.uint8))
    m = pf.Matcher(pf.Tables.from_bytes(long1 + b"\nab\n", 1, 256), device=0)
    with pytest.raises(pf.PfacError) as e:
        m.scan_batch(d, [0, 100, 500])
    assert e.value.code == PFAC_ERR_LIMIT
    assert len(m.scan_device(d)) == 200          # the context itself works ("ab" twice per "abcab")
    m.close()
    # 513 bytes are fine
    m = pf.Matcher(pf.Tables.from_bytes(long1[:513] + b"\nab\n", 1, 256), device=0)
    assert m.scan_batch(d, [0, 100, 500])[0].tolist() == [0, 40, 200]
    m.close()
    # DAG tables
    t = pf.Tables.from_bytes(b"abc\nacd\nbx\nab\n")
    p = t.part(0)
    s0 = p.s0.copy()
    s0[ord("b")] = s0[ord("a")]
    dag = pf.Tables.from_arrays(s0, p.r, p.HT, p.val, 256, p.state_num, p.n_final, p.idmap, p.max_len)
    m = pf.Matcher(dag, device=0)
    with pytest.raises(pf.PfacError) as e:
        m.scan_batch(d, [0, 500])
    assert e.value.code == PFAC_ERR_ARG
    m.close()
    # bad offsets, then the context still scans correctly
    pats = b"abcab\nab\nb\n"
    o = Oracle(pats, 1, 256)
    m = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256), device=0)
    for bad in ([1, 100, 500], [0, 300, 200, 500]):
        with pytest.raises(pf.PfacError) as e:
            m.scan_batch(d, bad)
        assert e.value.code == PFAC_ERR_ARG, bad
        check_batch(m, o, [b"abcab" * 20, b"", b"cabca" * 60])
    cnt = C.c_uint64(0)
    offs = np.array([0, 5], dtype=np.uint64)
    assert lib.pfac_scan_batch_device_sync(m._h, d.data_ptr(), None, 1, None, 0, d.data_ptr(), C.byref(cnt), None) == PFAC_ERR_ARG
    assert lib.pfac_scan_batch_device_sync(m._h, d.data_ptr(), offs.ctypes.data, 1, None, 0, None, C.byref(cnt), None) == PFAC_ERR_ARG
    m.close()
