"""Streaming scan of many flows (pfac_scan_flows_device_sync / Matcher.flows): the union of a flow's records over its
calls equals one scan of its whole stream, every record ends in the chunk that reported it, records of a chunk are
ordered by (pos, pattern length), and a call that does not fit or is refused leaves every flow unchanged."""
import ctypes as C

import numpy as np
import pytest

import phfpfac_b200 as pf
import pfac_synth as synth
from _oracle import Oracle
from phfpfac_b200._lib import PFAC_ERR_ARG, PFAC_ERR_LIMIT, PFAC_ERR_OUTPUT_FULL, lib
from test_detector_paths_host import CASES, get_case, phase_text, set_env
from test_flows_host import random_set

pytestmark = pytest.mark.gpu


def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


class Driver:
    """Feeds chunks to a Flows set, checks every call's records and collects them per flow."""

    def __init__(self, fs, lengths):
        self.fs, self.lengths = fs, np.asarray(lengths, dtype=np.int64)
        self.got = {}

    def call(self, items, **scan_kw):
        """items: [(flow, chunk bytes)] for distinct flows, one call."""
        before = {f: self.fs.position(f) for f, _ in items}
        if scan_kw:
            recs = self._scan(items, **scan_kw)
        else:
            recs = self.fs.feed([f for f, _ in items], [c for _, c in items])
        for (f, ch), r in zip(items, recs):
            P0, P1 = before[f], before[f] + len(ch)
            assert self.fs.position(f) == P1
            pos = r["pos"].astype(np.int64)
            L = self.lengths[r["id"].astype(np.int64)]
            assert ((pos + L > P0) & (pos + L <= P1)).all(), (f, P0, P1)
            key = list(zip(pos.tolist(), L.tolist()))
            assert key == sorted(key), f
            self.got.setdefault(f, []).append((pos, r["id"].astype(np.int32)))
        return recs

    def _scan(self, items, offset=0, cap=None):
        torch = torch_cuda()
        buf = np.concatenate([np.frombuffer(bytes(c), dtype=np.uint8) for _, c in items] + [np.zeros(0, np.uint8)])
        offs = np.zeros(len(items) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(c) for _, c in items])
        d = torch.zeros(offset + len(buf) + 16, dtype=torch.uint8, device="cuda")
        if len(buf):
            d[offset:offset + len(buf)] = torch.from_numpy(buf.copy()).cuda()
        first, base, rec = self.fs.scan([f for f, _ in items], d, offs, offset=offset, cap=cap)
        out = []
        for i in range(len(items)):
            seg = rec[int(first[i]):int(first[i + 1])]
            r = np.zeros(len(seg), dtype=pf.FLOW_MATCH_DTYPE)
            r["pos"], r["id"] = seg["pos"].astype(np.uint64) + base[i], seg["id"]
            out.append(r)
        return out

    def union(self, f):
        parts = self.got.get(f, [])
        pos = np.concatenate([p for p, _ in parts] + [np.zeros(0, np.int64)])
        ids = np.concatenate([i for _, i in parts] + [np.zeros(0, np.int32)])
        order = np.lexsort((self.lengths[ids.astype(np.int64)], pos))
        return pos[order], ids[order]

    def check(self, f, want, what=""):
        pos, ids = self.union(f)
        wp, wi = want
        assert len(pos) == len(wp), (what, f, len(pos), len(wp))
        assert np.array_equal(pos, np.asarray(wp, dtype=np.int64)) and np.array_equal(ids, np.asarray(wi, dtype=np.int32)), (what, f)


def feed_streams(drv, streams, sizes_of, rng, per_call):
    """Feed every flow's stream (dict flow -> bytes) in chunks whose sizes sizes_of(flow) yields, a random subset of
    at most per_call flows per call, until every stream is consumed."""
    at = {f: 0 for f in streams}
    gens = {f: sizes_of(f) for f in streams}
    while True:
        left = [f for f in streams if at[f] < len(streams[f])]
        if not left:
            return
        pick = rng.permutation(left)[:per_call]
        items = []
        for f in pick.tolist():
            s = next(gens[f])
            items.append((f, streams[f][at[f]:at[f] + s]))
            at[f] += s
        drv.call(items)


@pytest.mark.parametrize("seed", range(6))
def test_random_sets_and_streams(seed):
    """Pattern sets of test_random_batches' generators (max length <= 513), 50-200 flows with random streams, random
    subsets of flows per call, chunks of 0, 1, shortest - 1, M - 2, M - 1, M, 8191, 8192, 8193, 16385 and random
    sizes; per flow the union equals the oracle's scan of the whole stream."""
    rng = np.random.default_rng(2000 + seed)
    alpha = [2, 3, 4, 26, 200, 5][seed]
    max_len = min(int(rng.integers(1, [6, 12, 40, 20, 16, 513][seed] + 1)), 513)
    blob = random_set(rng, alpha, int(rng.integers(1, 2000)), max_len)
    t = pf.Tables.from_bytes(blob, 1, int(2 ** rng.integers(4, 13)))
    M = t.max_pat_len
    shortest = min(len(p) for p in blob.split(b"\n")[:-1])
    m = pf.Matcher(t, device=0)
    fs = m.flows(int(rng.integers(50, 201)))
    drv = Driver(fs, t.pattern_lengths())
    pool = [0, 1, max(shortest - 1, 0), max(M - 2, 0), max(M - 1, 0), M, 8191, 8192, 8193, 16385]

    def sizes_of(f):
        r = np.random.default_rng(seed * 1000 + f)
        while True:
            yield pool[int(r.integers(0, len(pool)))] if r.random() < 0.6 else int(r.integers(0, 3000))
    streams = {f: rng.integers(0, alpha, int(rng.integers(0, 40000))).astype(np.uint8).tobytes()
               for f in range(fs.n_flows)}
    feed_streams(drv, streams, sizes_of, rng, int(rng.integers(1, fs.n_flows + 1)))
    o = Oracle(blob, 1, 256)
    for f, s in streams.items():
        assert fs.position(f) == len(s)
        drv.check(f, o.scan(s), "random")
    m.close()


@pytest.mark.parametrize("name", list(CASES))
def test_every_kernel_path(name, monkeypatch):
    """The planted texts of the detector-path cases streamed by several flows, each cut next to every plant at a
    different offset into it, so plants straddle chunk borders at every offset; F2 (patterns of 900 B) and G (a
    DAG) are refused when the flow set is created."""
    torch_cuda()
    case = get_case(name)
    set_env(monkeypatch, case.spec)
    m = pf.Matcher(case.tables, device=0)
    if name == "F2":
        with pytest.raises(pf.PfacError) as e:
            m.flows(4)
        assert e.value.code == PFAC_ERR_LIMIT
        m.close()
        return
    if name == "G":
        with pytest.raises(pf.PfacError) as e:
            m.flows(4)
        assert e.value.code == PFAC_ERR_ARG
        m.close()
        return
    text, info = phase_text(case)
    want = case.reference(text)
    plants = info["plants"]
    span = case.max_len + 1
    data = text.tobytes()
    fs = m.flows(3)
    drv = Driver(fs, np.concatenate([[0], case.lens]))
    cuts = {}
    for f in range(3):
        c = sorted({min(len(data), a + (j * (2 * f + 1) + f) % span) for j, a in enumerate(plants)} | {len(data)})
        cuts[f] = c
    at = {f: 0 for f in range(3)}
    k = {f: 0 for f in range(3)}
    while any(at[f] < len(data) for f in range(3)):
        items = []
        for f in range(3):
            if at[f] < len(data):
                e = cuts[f][k[f]]
                items.append((f, data[at[f]:e]))
                at[f], k[f] = e, k[f] + 1
        drv.call(items)
        if len(items) == 3 and all(len(c) for _, c in items):
            assert m.last_info()["launches"] == 5 + case.spec["launches"], name
    for f in range(3):
        drv.check(f, want, name)
    m.close()


def oracle_driver(pats, n_flows=4):
    t = pf.Tables.from_bytes(pats, 1, 256)
    m = pf.Matcher(t, device=0)
    fs = m.flows(n_flows)
    return m, fs, Driver(fs, t.pattern_lengths()), Oracle(pats, 1, 256), t.max_pat_len


def test_needle_one_byte_per_call():
    m, fs, drv, o, M = oracle_driver(b"needle\nle\nneedles\nn\n")
    s = b"xxneedleneedlesxle" * 3
    for i in range(len(s)):
        recs = drv.call([(0, s[i:i + 1]), (1, s[:0])])
    drv.check(0, o.scan(s))
    assert fs.position(1) == 0 and len(drv.union(1)[0]) == 0
    m.close()


def test_longest_pattern_from_the_oldest_tail_byte():
    rng = np.random.default_rng(9)
    P = bytes(rng.integers(97, 123, 40).astype(np.uint8))
    m, fs, drv, o, M = oracle_driver(P + b"\nab\n" + P[:7] + b"\n")
    assert M == 40
    # flow 0: the tail holds exactly P[:M-1] after junk; flow 1: the stream so far is exactly M - 1 bytes
    recs = drv.call([(0, b"q" * 100 + P[:M - 1]), (1, P[:M - 1])])
    recs = drv.call([(0, P[M - 1:]), (1, P[M - 1:])])
    for f, start in ((0, 100), (1, 0)):
        full = recs[f][recs[f]["id"] == 1]
        assert full["pos"].tolist() == [start], f
    drv.check(0, o.scan(b"q" * 100 + P))
    drv.check(1, o.scan(P))
    m.close()


def test_match_ending_at_a_chunk_end_is_reported_once():
    m, fs, drv, o, M = oracle_driver(b"needle\nle\nneedlexyz\n")
    recs = drv.call([(0, b"xxneedle")])
    assert recs[0]["pos"].tolist() == [2, 6]
    for ch in (b"", b"x", b"", b"y", b"q"):
        recs = drv.call([(0, ch)])
        assert len(recs[0]) == 0
    drv.check(0, o.scan(b"xxneedlexyq"))
    m.close()


def test_flow_shorter_than_the_tail_for_many_calls():
    rng = np.random.default_rng(4)
    pats = random_set(rng, 3, 200, 6) + bytes(rng.integers(97, 100, 60).astype(np.uint8)) + b"\n"
    alphabet = sorted(set(pats) - {10})
    m, fs, drv, o, M = oracle_driver(pats)
    assert M == 60
    s = bytes(rng.choice(alphabet, 57).astype(np.uint8).tolist())
    at = 0
    while at < len(s):
        n = int(rng.integers(0, 3))
        drv.call([(2, s[at:at + n])])
        at += n
        assert fs.position(2) == min(at, len(s)) < M - 1
    drv.check(2, o.scan(s))
    assert len(drv.union(2)[0]) > 10
    m.close()


@pytest.mark.parametrize("offset", (0, 1, 2, 3, 7, 8, 15))
def test_misaligned_chunks_and_lengths_around_16_byte_phases(offset):
    pats = b"abcab\nab\nb\ncabcabcabc\nabcabcabcabcabcabcabcabcabcabcabcab\nbca\n"
    m, fs, drv, o, M = oracle_driver(pats, n_flows=70)
    rng = np.random.default_rng(offset)
    base = (b"abc" * 400 + b"ab" * 200) * 4
    streams = {f: b"" for f in range(70)}
    for rnd in range(6):
        items = []
        for f in range(70):
            n = (f + 7 * rnd) % 64 + 1
            a = int(rng.integers(0, len(base) - n))
            items.append((f, base[a:a + n]))
            streams[f] += base[a:a + n]
        drv.call(items, offset=offset)
    for f, s in streams.items():
        drv.check(f, o.scan(s), offset)
    m.close()


def test_one_64_mib_chunk():
    torch = torch_cuda()
    pats = synth.synth_patterns(1, 2000, 13, 4, 48)
    t = pf.Tables.from_bytes(pats, 1, 256)
    m = pf.Matcher(t, device=0)
    fs = m.flows(2)
    drv = Driver(fs, t.pattern_lengths())
    text = synth.synth_text(1, 14, (64 << 20) + 5000, patterns=pats)
    head, big = text[:5000].tobytes(), text[5000:]
    drv.call([(1, head)])
    drv.call([(1, big)], offset=3)
    want = m.scan_device(torch.from_numpy(text.copy()).cuda(), cap=len(text) // 16)
    assert len(want) > 1000
    drv.check(1, (want["pos"].astype(np.int64), want["id"].astype(np.int32)))
    m.close()


def test_100000_packets_in_one_call():
    """Two calls of 100,000 packets of 40-1500 B, one per flow; per flow the union equals the batch scan of the
    flow's two packets concatenated."""
    torch = torch_cuda()
    pats = synth.synth_patterns(1, 3000, 17, 4, 64)
    t = pf.Tables.from_bytes(pats, 1, 256)
    lengths = t.pattern_lengths().astype(np.int64)
    m = pf.Matcher(t, device=0)
    n = 100000
    fs = m.flows(n)
    rng = np.random.default_rng(6)
    sizes = rng.integers(40, 1501, (2, n))
    text = synth.synth_text(1, 18, int(sizes.sum()) + 1, patterns=pats)
    got = []
    at = 0
    flows = [rng.permutation(n).astype(np.uint32), rng.permutation(n).astype(np.uint32)]
    starts = np.zeros((2, n), dtype=np.int64)
    for c in range(2):
        offs = np.zeros(n + 1, dtype=np.uint64)
        offs[1:] = np.cumsum(sizes[c][flows[c]])
        starts[c][flows[c]] = at + offs[:-1].astype(np.int64)
        d = torch.from_numpy(text[at:at + int(offs[-1])].copy()).cuda()
        first, base, rec = fs.scan(flows[c], d, offs)
        chunk = np.repeat(np.arange(n), np.diff(first.astype(np.int64)))
        got.append((flows[c][chunk].astype(np.int64), rec["pos"].astype(np.int64) + base[chunk].astype(np.int64),
                    rec["id"].astype(np.int64)))
        at += int(offs[-1])
    assert all(fs.position(f) == int(sizes[0][f] + sizes[1][f]) for f in range(0, n, 997))
    # reference: each flow's stream as one document of a batch
    docs = np.concatenate([np.concatenate([text[starts[0][f]:starts[0][f] + sizes[0][f]],
                                           text[starts[1][f]:starts[1][f] + sizes[1][f]]]) for f in range(n)])
    doffs = np.zeros(n + 1, dtype=np.uint64)
    doffs[1:] = np.cumsum(sizes[0] + sizes[1])
    wfirst, wrec = m.scan_batch(docs, doffs)
    wflow = np.repeat(np.arange(n), np.diff(wfirst.astype(np.int64)))
    gf = np.concatenate([g[0] for g in got])
    gp = np.concatenate([g[1] for g in got])
    gi = np.concatenate([g[2] for g in got])
    order = np.lexsort((lengths[gi], gp, gf))
    assert len(gf) == len(wrec) > 1000
    assert np.array_equal(gf[order], wflow) and np.array_equal(gp[order], wrec["pos"].astype(np.int64))
    assert np.array_equal(gi[order], wrec["id"].astype(np.int64))
    m.close()


def raw_call(fs, d, offs, ids, cap):
    torch = torch_cuda()
    out = torch.full((cap + 64, 2), 0x5a5a5a5a, dtype=torch.int32, device="cuda")
    first = torch.zeros(len(ids) + 1, dtype=torch.int64, device="cuda")
    base = np.zeros(max(len(ids), 1), dtype=np.uint64)
    cnt = C.c_uint64(0)
    rc = lib.pfac_scan_flows_device_sync(fs._h, d.data_ptr(), offs.ctypes.data, ids.ctypes.data, len(ids), out.data_ptr(),
                                         cap, first.data_ptr(), base.ctypes.data, C.byref(cnt), None)
    return rc, cnt.value, out


@pytest.mark.parametrize("pats", [b"needle\nle\nneedlework\nwork\n", b"a\naa\naaa\nb\n"])
def test_output_full_commits_nothing(pats):
    """cap below the count (and, for the dense set, below the raw records too): OUTPUT_FULL, positions and tails
    unchanged; the rescan with the returned count and every later call equal a run that never overflowed."""
    torch = torch_cuda()
    m, fs, drv, o, M = oracle_driver(pats, n_flows=3)
    ref = Driver(m.flows(3), drv.lengths)
    rng = np.random.default_rng(8)
    dense = b"needle" not in pats
    alphabet = b"aab" if dense else b"needlwork"
    streams = {f: b"" for f in range(3)}
    raw_overflow = False
    for rnd in range(8):
        items = [(f, bytes(rng.choice(list(alphabet), int(rng.integers(0, 9000))).astype(np.uint8).tolist()))
                 for f in range(3)]
        ref.call(items)
        buf = b"".join(c for _, c in items)
        offs = np.zeros(4, dtype=np.uint64)
        offs[1:] = np.cumsum([len(c) for _, c in items])
        ids = np.arange(3, dtype=np.uint32)
        d = torch.from_numpy(np.frombuffer(buf + b"\0" * 16, dtype=np.uint8).copy()).cuda()
        want = sum(len(r[0]) for r in (ref.got[f][-1] for f in range(3)))
        if want > 1:
            before = [fs.position(f) for f in range(3)]
            cap = int(rng.integers(0, min(want, 4096)))
            rc, cnt, out = raw_call(fs, d, offs, ids, cap)
            assert rc == PFAC_ERR_OUTPUT_FULL and cnt >= want, (cap, cnt, want)
            assert (out[cap:] == 0x5a5a5a5a).all().item()
            assert [fs.position(f) for f in range(3)] == before
            raw_overflow |= want > 4096     # (the raw buffer holds max(cap, 4096) records: the raw count is passed on)
            recs = drv.call(items, cap=cnt)  # the rescan with the returned count fits at once
        else:
            recs = drv.call(items)
        for f, (_, c) in enumerate(items):
            streams[f] += c
            assert np.array_equal(recs[f]["pos"].astype(np.int64), ref.got[f][-1][0])
            assert np.array_equal(recs[f]["id"].astype(np.int32), ref.got[f][-1][1])
    assert raw_overflow == dense
    for f in range(3):
        drv.check(f, o.scan(streams[f]))
    m.close()


def test_reset_and_refusals_leave_state_unchanged():
    torch = torch_cuda()
    m, fs, drv, o, M = oracle_driver(b"needle\nle\nhaystack\n", n_flows=4)
    drv.call([(0, b"xxnee"), (1, b"hays")])
    fs.reset(0)
    assert fs.position(0) == 0
    recs = drv.call([(0, b"dlexx"), (1, b"tack")])
    assert recs[0]["pos"].tolist() == [1] and recs[1]["pos"].tolist() == [0]   # "le" only; haystack straddles
    d = torch.from_numpy(np.frombuffer(b"needle" * 10, dtype=np.uint8).copy()).cuda()
    bad = [([0, 0], [0, 6, 12]), ([0, 4], [0, 6, 12]), ([1, 2], [1, 6, 12]), ([1, 2], [0, 12, 6])]
    for ids, offs in bad:
        before = [fs.position(f) for f in range(4)]
        with pytest.raises(pf.PfacError) as e:
            fs.scan(ids, d, offs)
        assert e.value.code == PFAC_ERR_ARG, (ids, offs)
        assert [fs.position(f) for f in range(4)] == before
    cnt = C.c_uint64(0)
    offs = np.array([0, 6], dtype=np.uint64)
    ids = np.array([0], dtype=np.uint32)
    assert lib.pfac_scan_flows_device_sync(fs._h, d.data_ptr(), offs.ctypes.data, None, 1, None, 0, d.data_ptr(), None,
                                           C.byref(cnt), None) == PFAC_ERR_ARG
    assert lib.pfac_flows_reset(fs._h, 4) == PFAC_ERR_ARG
    drv.call([(0, b"needle"), (1, b"needle")])
    drv.check(0, o.scan(b"dlexxneedle"))
    drv.check(1, o.scan(b"haystackneedle"))
    m.close()
    assert fs._h is None        # Matcher.close() closed its flow set first


def test_interleaved_with_device_and_batch_scans_and_streams(fixtures):
    torch = torch_cuda()
    pats = fixtures["xac"]
    o = Oracle(pats, 1, 256)
    t = pf.Tables.from_bytes(pats, 1, 256)
    m = pf.Matcher(t, device=0)
    fs = m.flows(20)
    drv = Driver(fs, t.pattern_lengths())
    base = np.frombuffer(fixtures["1M"], dtype=np.uint8)
    whole = base[:300000].copy()
    want_whole = o.scan(whole)
    d_whole = torch.from_numpy(whole).cuda()
    docs = [base[i * 1000:i * 1000 + 700].tobytes() for i in range(50)]
    want_docs = [o.scan(x) for x in docs]
    streams = {f: b"" for f in range(20)}
    rng = np.random.default_rng(12)
    launches = 6 if m.derived_info()["has_short"] else 8   # (patterns of <= 3 bytes: the dense-match kernel alone)
    streams_t = [torch.cuda.current_stream(), torch.cuda.Stream(), torch.cuda.Stream()]
    for rep in range(9):
        with torch.cuda.stream(streams_t[rep % 3]):
            items = []
            for f in rng.permutation(20)[:12].tolist():
                a = int(rng.integers(0, len(base) - 5000))
                items.append((f, base[a:a + int(rng.integers(0, 5000))].tobytes()))
                streams[f] += items[-1][1]
            drv.call(items)
            info = m.last_info()
            assert info["launches"] == launches and info["h2d_bytes"] == 4 * (4 * len(items) + 1)
            got = m.scan_device(d_whole)
            assert np.array_equal(got["pos"].astype(np.int64), want_whole[0])
            for w, r in zip(want_docs, m.scan_docs(docs)):
                assert np.array_equal(r["pos"].astype(np.int64), w[0]) and np.array_equal(r["id"].astype(np.int32), w[1])
    for f in range(20):
        drv.check(f, o.scan(streams[f]))
    m.close()


def test_direct_set_launches_and_one_byte_patterns():
    """A set with patterns of <= 3 bytes runs the dense-match kernel alone (6 launches); a set of 1-byte patterns
    carries nothing and behaves like a batch."""
    for pats, launches in ((b"a\nab\nabc\nbca\n", 6), (b"a\nb\nc\n", 6)):
        m, fs, drv, o, M = oracle_driver(pats, n_flows=5)
        rng = np.random.default_rng(len(pats))
        streams = {f: b"" for f in range(5)}
        for rnd in range(10):
            items = [(f, bytes(rng.choice(list(b"abcx"), int(rng.integers(1, 300))).astype(np.uint8).tolist()))
                     for f in range(5)]
            drv.call(items)
            assert m.last_info()["launches"] == launches
            for f, c in items:
                streams[f] += c
        for f in range(5):
            drv.check(f, o.scan(streams[f]))
        m.close()
