"""Every scan entry point against the sparse reference above 2 GiB: single calls at the 4 GiB limit, batches and flows
whose positions pass 2^31 and 2^32, jobs and the CLI past 4 GiB.  Layouts and references:
tests/test_large_inputs_host.py.  Inputs are views of one device buffer of background bytes (2^32 + 64 bytes) with
plants written in and taken out again; every call passes an explicit record capacity."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import phfpfac_b200 as pf
import pfac_synth as synth
from _oracle import Oracle, render_result
from phfpfac_b200._lib import PFAC_ERR_LIMIT, lib
from test_detector_paths_gpu import check_signature
from test_detector_paths_host import BG, TILE, get_case, set_env
from test_large_inputs_host import (LARGE_CASES, Plants, Reference, case_reference, flow_case, flow_view,
                                    max_call_bytes, scan_layout, seam_split, small_plants, straddler, stream_reference)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GPHF = os.path.join(ROOT, "phfpfac_b200", "_build", "gphf")
BUF_BYTES = 2 ** 32 + 64
G31, G32 = 1 << 31, 1 << 32


@pytest.fixture(scope="session")
def big():
    """The device buffer, all background; tests write plants into it and restore the background afterwards."""
    import torch
    assert torch.cuda.is_available()
    buf = DeviceText(torch.full((BUF_BYTES,), BG, dtype=torch.uint8, device="cuda"))
    yield buf
    del buf.t
    torch.cuda.empty_cache()


class DeviceText:
    def __init__(self, t):
        self.t = t
        self.written = []

    def write(self, plants, origin=0):
        """The clusters of `plants` at buffer offset origin + position."""
        import torch
        small_idx, small_val = [], []
        for s, b in plants:
            a = origin + s
            assert 0 <= a and a + len(b) <= BUF_BYTES
            v = np.frombuffer(b, dtype=np.uint8)
            if len(b) > 4096:
                self.t[a:a + len(b)].copy_(torch.from_numpy(v.copy()))
                self.written.append((a, len(b)))
            else:
                small_idx.append(np.arange(a, a + len(b), dtype=np.int64))
                small_val.append(v)
        if small_idx:
            idx = torch.from_numpy(np.concatenate(small_idx)).cuda()
            self.t[idx] = torch.from_numpy(np.concatenate(small_val)).cuda()
            self.written.append(idx)
        torch.cuda.synchronize()

    def restore(self):
        for w in self.written:
            if isinstance(w, tuple):
                self.t[w[0]:w[0] + w[1]].fill_(BG)
            else:
                self.t[w] = BG
        self.written = []
        import torch
        torch.cuda.synchronize()


def same(got, want, what):
    pos, ids = want
    assert len(got) == len(pos), (what, len(got), len(pos))
    assert np.array_equal(got["pos"].astype(np.int64), pos), what
    assert np.array_equal(got["id"].astype(np.int32), ids), what


def limit_refused(fn):
    with pytest.raises(pf.PfacError) as e:
        fn()
    assert e.value.code == PFAC_ERR_LIMIT, e.value


# ---------------------------------------------------------------- a. scan_device at and around the limit

@pytest.mark.parametrize("name", LARGE_CASES)
def test_scan_device_at_the_limit(big, name, monkeypatch):
    """n = 2^31 (256 tiles per ordering CTA), 2^31 + 1 (257: the first size whose chunk loop repeats) and the largest
    size a call accepts, at pointer offsets 0 and 15: plants across 2^31, the phase block (every plant at the lane,
    slot and tile phases, tiles of 1, 2, 3-32 and more than 32 plants, near-misses), plants in the first and the
    second 256-tile chunk of ordering CTAs' ranges, the end zone; n_starts < n_valid and a pattern cut by n_valid at
    the top.  One byte more than the largest size is refused."""
    case = get_case(name)
    set_env(monkeypatch, case.spec)
    ref = case_reference(case)
    m = pf.Matcher(case.tables, device=0, n_streams=2)
    check_signature(m, case)
    d = big.t
    s_len = len(straddler(case))
    k = 0
    for mis in (0, 15):
        top = max_call_bytes(mis)
        for n in (G31, G31 + 1, top):
            k += 1
            bases = [0] + ([(1 << 32) + 4096 * 7 + 1234] if case.max_len > 513 and n == top else [])
            for base_pos in bases:
                P, info = scan_layout(case, n, mis, base_pos=base_pos, straddle=1 + (7 * k) % (s_len - 1))
                big.write(P, mis)
                try:
                    runs = [(n, n)]
                    if info["end"] is not None:
                        runs += [(info["end"], n), (info["end"] + 1, n), (n - 1, n - 1)]
                    for ns, nv in runs:
                        want = ref(P, 0, nv, ns, base_pos=base_pos)
                        got = m.scan_device(d, n_starts=ns, n_valid=nv, base_pos=base_pos, offset=mis, cap=len(want[0]) + 1024)
                        same(got, want, (name, mis, n, base_pos, ns, nv))
                        info_ = m.last_info()
                        assert info_["tiles"] == -(-(mis + ns) // TILE) and info_["launches"] == case.spec["launches"]
                    if n == top:
                        assert (want[0] >= G31).sum() > 100
                finally:
                    big.restore()
        limit_refused(lambda: m.scan_device(d, n_starts=top + 1, n_valid=top + 1, offset=mis, cap=1024))
        # n_valid past the limit is accepted when the starts leave it unused (n_valid is cut to n_starts + M - 1)
        ns = top - case.max_len + 1
        assert len(m.scan_device(d, n_starts=ns, n_valid=BUF_BYTES - mis, offset=mis, cap=1024)) == 0
        limit_refused(lambda: m.scan_device(d, n_starts=ns + 1, n_valid=BUF_BYTES - mis, offset=mis, cap=1024))
    m.close()


@pytest.mark.parametrize("name", ["A", "H", "J3"])
def test_scan_device_straddles_2_31_at_every_offset(big, name, monkeypatch):
    """The straddler across 2^31 with 1 .. len - 1 of its bytes below it, one scan each."""
    case = get_case(name)
    set_env(monkeypatch, case.spec)
    ref = case_reference(case)
    m = pf.Matcher(case.tables, device=0, n_streams=2)
    s = straddler(case)
    n = G31 + 4096
    for j in range(1, len(s)):
        P = Plants(case.max_len)
        P.must_put(G31 - j, s)
        big.write(P)
        try:
            want = ref(P, 0, n)
            assert len(want[0]) >= 1
            same(m.scan_device(big.t, n_starts=n, n_valid=n, cap=1024), want, (name, j))
        finally:
            big.restore()
    m.close()


# ---------------------------------------------------------------- b. real text above 2 GiB

def test_real_text_above_2_GiB(big):
    """Config-3-shaped patterns over 3 GiB + 12,345 bytes of synthetic text: one scan_device equals the concatenation
    of four shards cut like plan_shard, the oracle on 1 MiB windows at 2^31 - 2^19, 2^31 and the end, and scan_host
    of the same array."""
    import torch
    pats = synth.synth_patterns(1, 10000, 3, 4, 64)
    t = pf.Tables.from_bytes(pats, 1, 256)
    lens = t.pattern_lengths().astype(np.int64)
    n = 3 * (1 << 30) + 12345
    text = synth.synth_text(1, 31, n, patterns=pats)
    d = big.t
    d[:n].copy_(torch.from_numpy(text))
    torch.cuda.synchronize()
    try:
        m = pf.Matcher(t, device=0)
        whole = m.scan_device(d, n_starts=n, n_valid=n, cap=n // 64)
        assert len(whole) > 1000 and (whole["pos"].astype(np.int64) >= G31).sum() > 100
        parts = []
        for i in range(4):
            a, ns, nv = pf.plan_shard(n, 4, t.max_pat_len, i)
            assert nv < (1 << 30)
            r = m.scan_device(d, n_starts=ns, n_valid=nv, base_pos=a, offset=a, cap=max(1024, ns // 64))
            parts.append(np.stack([r["pos"].astype(np.int64) + a, r["id"].astype(np.int64)], 1))
        cat = np.concatenate(parts)
        assert np.array_equal(cat[:, 0], whole["pos"].astype(np.int64)) and np.array_equal(cat[:, 1], whole["id"].astype(np.int64))
        o = Oracle(pats, 1, 256)
        wp, wi = whole["pos"].astype(np.int64), whole["id"].astype(np.int64)
        wend = wp + lens[wi]
        for w in (G31 - (1 << 19), G31, n - (1 << 20)):
            pos, ids = o.scan(text[w:w + (1 << 20)])
            keep = (wp >= w) & (wend <= w + (1 << 20))
            assert len(pos) > 0 and np.array_equal(wp[keep] - w, pos) and np.array_equal(wi[keep], ids), w
        host = m.scan_host(text, cap=len(whole) + 1024)
        assert np.array_equal(host, whole)
        m.close()
    finally:
        big.t[:n].fill_(BG)
        torch.cuda.synchronize()


# ---------------------------------------------------------------- c. scan_host at n_valid = 2^32 - 1

def test_scan_host_at_4_GiB():
    """A host array of 2^32 - 1 bytes: sub-chunks whose pos_bias approaches 2^32, records past 2^31, plants across
    sub-chunk borders (default chunk size and one that is not a multiple of the tile, which the context rounds up),
    a pattern ending at the last byte.  n_valid = 2^32 is refused."""
    case = get_case("A")
    ref = case_reference(case)
    n = G32 - 1
    s = straddler(case)
    fill = small_plants(case)
    chunks = [32 << 20, 3 * TILE * 1000 + 5]
    P = Plants(case.max_len)
    for c in chunks:
        c_eff = -(-c // TILE) * TILE
        for b in sorted({c_eff, G31 // c_eff * c_eff, (G31 // c_eff + 1) * c_eff, (n // c_eff) * c_eff,
                         (n // c_eff - 1) * c_eff}):
            for j, d in enumerate((1, len(s) // 2, len(s) - 1)):
                P.put(b - d + j * 8 * TILE, s)
    for k in range(200):
        P.put(G31 + k * 7919 * 1013 + k, fill[k % len(fill)])
    last = fill[3]
    P.must_put(n - len(last), last)
    text = P.text(0, n)
    want = ref(P, 0, n)
    assert (want[0] >= G31).sum() > 100 and want[0][-1] == n - len(last)
    for c in (0, chunks[1]):
        m = pf.Matcher(case.tables, device=0, n_streams=3, chunk_bytes=c)
        same(m.scan_host(text, cap=len(want[0]) + 1024), want, ("host", c))
        out = np.zeros(16, dtype=pf.MATCH_DTYPE)
        cnt = C.c_uint64(0)
        assert lib.pfac_scan_host(m._h, text.ctypes.data, G32, G32, 0, out.ctypes.data, 16, C.byref(cnt)) == PFAC_ERR_LIMIT
        m.close()


# ---------------------------------------------------------------- d. batch above 2 GiB

def test_batch_above_2_GiB(big):
    """Documents as views of the buffer: boundaries at 2^31 - 1, 2^31 and 2^31 + 1, empty documents at 2^31,
    thousands of small documents past 2^31 with plants across their ends, one document larger than 2 GiB.  Each
    document's records equal the sparse reference of that document alone; a total of max_call_bytes(mis) is
    accepted and one byte more is refused."""
    case = get_case("A")
    ref = case_reference(case)
    m = pf.Matcher(case.tables, device=0)
    rng = np.random.default_rng(7)
    s = straddler(case)
    fill = small_plants(case)
    for mis, layout in ((0, "big document"), (15, "boundaries")):
        total = max_call_bytes(mis)
        if layout == "big document":
            offs = [0, 1000, G31 + (3 << 20)] + [G31 + (3 << 20) + 5000 * i for i in range(1, 6)] + [total]
        else:
            offs = [0, G31 - 1, G31, G31, G31, G31, G31 + 1]
            at = G31 + 1
            for _ in range(4000):
                at += int(rng.integers(1, 3000))
                offs.append(at)
            offs.append(total)
        offs = np.array(offs, dtype=np.uint64)
        P = Plants(case.max_len)
        for i, b in enumerate(offs[1:-1].tolist()):      # across document ends, ending on them, inside documents
            P.put(b - 1 - i % (len(s) - 1), s) or P.put(b - len(fill[i % 7]), fill[i % 7]) or P.put(b + 3, fill[i % 5])
        for k in range(300):
            P.put(int(rng.integers(0, total - 100)), fill[k % len(fill)])
        last = fill[2]
        P.put(total - len(last), last)
        big.write(P, mis)
        try:
            first, rec = m.scan_batch(big.t, offs, offset=mis, cap=len(P.starts) * 8 + 4096)
            assert len(first) == len(offs)
            allp, n_past = 0, 0
            for i in range(len(offs) - 1):
                a, b = int(offs[i]), int(offs[i + 1])
                want = ref(P, a, b - a)
                same(rec[int(first[i]):int(first[i + 1])], want, (mis, i, a, b))
                allp += len(want[0])
                n_past += int((want[0] + a >= G31).sum())
            assert int(first[-1]) == allp and allp > 100 and n_past > 50
            if layout == "big document":
                assert int(first[2]) - int(first[1]) > 10      # the document of more than 2 GiB
        finally:
            big.restore()
        over = offs.copy()
        over[-1] += 1
        limit_refused(lambda: m.scan_batch(big.t, over, offset=mis, cap=4096))
    m.close()


# ---------------------------------------------------------------- e. flows past 2^32

def test_flows_past_4_GiB(big):
    """Three flows fed more than 5 GiB each in calls of about 1 GiB per flow, all views of the buffer: flow 0 has a
    seam exactly at stream position 2^32 (a match ends there, one starts there, two cross it), flow 1 crosses 2^32
    mid-chunk, flow 2 has chunks of 2^30 + 4097 bytes.  Absolute positions, position() and each flow's union equal
    the stream model.  A call whose chunks are below the limit but whose chunks plus carried tails reach it is
    refused and changes no position; one byte less passes."""
    case = flow_case()
    split = seam_split(case)
    assert split is not None
    S, j = split
    m = pf.Matcher(case.tables, device=0)
    fs = m.flows(3)
    lens = case.lens
    sizes = [1 << 30, (1 << 30) - 12345, (1 << 30) + 4097]
    o = 5
    starts = [o, o + sizes[0], o + sizes[0] + sizes[1]]
    # flow 1: the view holds a plant across the stream position 2^32, which its 5th chunk reaches mid-chunk
    k1 = G32 // sizes[1]
    mid1 = G32 - k1 * sizes[1]
    assert 0 < mid1 < sizes[1]
    inner = [(1000, 500000, sizes[0] // 2), (mid1 - 3, 77777, sizes[1] - 9999), (123457, sizes[2] - 88888)]
    P = None
    for f in range(3):
        V = flow_view(case, sizes[f], split, inner[f]).shifted(starts[f])
        P = V if P is None else P.merged(V)
    big.write(P)
    views = {f: [] for f in range(3)}
    got = {f: [] for f in range(3)}
    try:
        n_calls = 6
        offs = np.array([0, sizes[0], sizes[0] + sizes[1], sum(sizes)], dtype=np.uint64)
        for call in range(n_calls):
            first, base, rec = fs.scan([0, 1, 2], big.t, offs, offset=o, cap=1 << 16)
            for f in range(3):
                seg = rec[int(first[f]):int(first[f + 1])]
                pos = seg["pos"].astype(np.int64) + int(base[f])
                P0 = call * sizes[f]
                ends = pos + lens[seg["id"].astype(np.int64) - 1]
                assert ((ends > P0) & (ends <= P0 + sizes[f])).all(), (call, f)
                got[f].append((pos, seg["id"].astype(np.int32)))
                views[f].append((starts[f], sizes[f]))
                assert fs.position(f) == (call + 1) * sizes[f]
        # the final call: chunks plus carried tails reach the limit by one byte, then one byte less
        carried = 3 * (case.max_len - 1)
        total = max_call_bytes(0) + 1 - carried
        assert total < max_call_bytes(0)
        cuts = [0, 1 << 30, 1 << 31, total]
        before = [fs.position(f) for f in range(3)]
        limit_refused(lambda: fs.scan([0, 1, 2], big.t, np.array(cuts, dtype=np.uint64), cap=1 << 16))
        assert [fs.position(f) for f in range(3)] == before
        cuts[-1] -= 1
        first, base, rec = fs.scan([0, 1, 2], big.t, np.array(cuts, dtype=np.uint64), cap=1 << 16)
        for f in range(3):
            seg = rec[int(first[f]):int(first[f + 1])]
            got[f].append((seg["pos"].astype(np.int64) + int(base[f]), seg["id"].astype(np.int32)))
            views[f].append((cuts[f], cuts[f + 1] - cuts[f]))
            assert fs.position(f) == before[f] + cuts[f + 1] - cuts[f]
    finally:
        big.restore()
    for f in range(3):
        pos = np.concatenate([p for p, _ in got[f]])
        ids = np.concatenate([i for _, i in got[f]])
        order = np.lexsort((lens[ids - 1], pos))
        want = stream_reference(case, P, views[f])
        assert len(pos) == len(want[0]) and np.array_equal(pos[order], want[0]) and np.array_equal(ids[order], want[1]), f
        assert want[0][-1] > 5 * (1 << 30)
    # flow 0's seam at 2^32: S across it, a match ending on it and one starting on it
    pos0 = np.concatenate([p for p, _ in got[0]])
    ids0 = np.concatenate([i for _, i in got[0]])
    assert ((pos0 == G32 - j) & (lens[ids0 - 1] == len(S))).any()
    assert (pos0 + lens[ids0 - 1] == G32).any() and (pos0 == G32).any()
    # flow 1: the plant across 2^32, mid-chunk
    pos1 = np.concatenate([p for p, _ in got[1]])
    ids1 = np.concatenate([i for _, i in got[1]])
    assert ((pos1 == G32 - 3) & (pos1 + lens[ids1 - 1] > G32)).any()
    fs.close()
    m.close()


# ---------------------------------------------------------------- f. job and CLI past 4 GiB

def test_job_past_4_GiB():
    """Job([0]) and Job(all devices) over a host array of 4 GiB + 3 MiB + 17 bytes: segment bases reach 4 GiB, a
    plant straddles each segment and shard border (2^32 among them), a pattern ends at n; global positions equal the
    sparse reference."""
    case = get_case("A")
    ref = case_reference(case)
    n = G32 + (3 << 20) + 17
    s = straddler(case)
    P = Plants(case.max_len)
    nd = pf.device_count()
    borders = {k << 30 for k in range(1, 5)}
    for nsh in {1, nd}:
        borders |= {pf.plan_shard(n, nsh, case.max_len, i)[0] for i in range(1, nsh)}
    for i, b in enumerate(sorted(borders)):
        if 0 < b < n - 100:
            P.put(b - 1 - i % (len(s) - 1), s)
    last = small_plants(case)[4]
    P.must_put(n - len(last), last)
    text = P.text(0, n)
    want = ref(P, 0, n)
    assert want[0][-1] == n - len(last) and (want[0] > G32 - len(s)).sum() >= 2
    for devices in ([0], list(range(nd))):
        job = pf.Job(case.tables, devices=devices, streams_per_gpu=4)
        total, segs = job.run(text)
        assert max(b for b, _ in segs) >= G32 or len(devices) > 1
        gp = np.concatenate([r[:, 0].astype(np.int64) + b for b, r in segs])
        gi = np.concatenate([r[:, 1].astype(np.int32) for b, r in segs])
        assert total == len(want[0]) and np.array_equal(gp, want[0]) and np.array_equal(gi, want[1]), devices
        job.close()


def test_job_file_and_cli_past_4_GiB(tmp_path):
    """run_file and gphf on a sparse file of 4 GiB + 3 MiB + 18 bytes (holes read as zero bytes; the set is A's lines
    without byte 0): GPU_match_result.txt carries positions above 2^32 and equals the reference's rendering."""
    base = get_case("A")
    blob = b"".join(p + b"\n" for p in base.lines if 0 not in p)
    o = Oracle(blob, 1, 256)
    lens = np.array([len(p) for p in blob.split(b"\n")[:-1]], dtype=np.int64)
    ref = Reference(o.scan, bg=0)
    n = G32 + (3 << 20) + 17
    lines = blob.split(b"\n")[:-1]
    s = max((p for p in lines if len(p) <= 64), key=len)
    P = Plants(int(lens.max()), bg=0)
    for i, b in enumerate((1 << 30, 1 << 31, 3 << 30, G32, G32 + (64 << 20), G32 + (2 << 20))):
        P.must_put(b - 1 - 3 * i, s)
    P.must_put(n - len(lines[7]), lines[7])
    path = tmp_path / "big.bin"
    with open(path, "wb") as f:
        os.truncate(f.fileno(), n + 1)
        for at, b in P:
            os.pwrite(f.fileno(), b, at)
    if os.stat(path).st_blocks * 512 > (64 << 20):
        pytest.skip("the filesystem of the temporary directory does not keep the file sparse")
    pos, ids = ref(P, 0, n)
    assert (pos >= G32).sum() >= 2 and (pos > G32 - len(s)).sum() >= 3 and pos[-1] == n - len(lines[7])
    t = pf.Tables.from_bytes(blob, 1, 256)
    job = pf.Job(t, devices=[0], streams_per_gpu=3)
    nm, segs = job.run_file(str(path), n)
    gp = np.concatenate([r[:, 0].astype(np.int64) + b for b, r in segs])
    gi = np.concatenate([r[:, 1].astype(np.int32) for b, r in segs])
    assert nm == len(pos) and np.array_equal(gp, pos) and np.array_equal(gi, ids)
    job.close()
    pat = tmp_path / "patterns"
    pat.write_bytes(blob)
    r = subprocess.run([GPHF, str(pat), "2", "256", str(path)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "GPU_match_result.txt").read_bytes() == render_result(pos, ids)
