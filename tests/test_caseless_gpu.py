"""Caseless pattern sets on the B200: every scan entry point of a set built with caseless=True returns, record for
record, what the oracle returns for the folded patterns over the folded text (tests/test_caseless_host.py).  The
device folds the text before the unchanged detector: the caller's bytes are never written, the fold is one more
launch per scan, and the tile geometry and size bounds are those of a case-sensitive call."""
import os
import subprocess

import numpy as np
import pytest

import phfpfac_b200 as pf
from _oracle import Oracle
from _caseless_ref import fold
from test_caseless_host import CASELESS_CASES, caseless_case, random_case
from test_detector_paths_gpu import Expect, check_signature, same
from test_detector_paths_host import BG, TILE, phase_text, set_env

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GPHF = os.path.join(ROOT, "phfpfac_b200", "_build", "gphf")


def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def mixed_set(seed):
    """Snort-like patterns in random case, HTTP words that collide after folding, and patterns of bytes 0xC1-0xDA
    (which must not fold)."""
    from pfac_synth import synth_patterns
    pats = synth_patterns(seed, 1500, 100 + seed, 4, 40)
    pats += b"GET /\nget /\nHost: \nContent-Length: \nUser-Agent: Mozilla\n\xc1\xc2\xd0\xda\n\xc1bc\xda\nAbC\xc1\n"
    return random_case(pats, seed)


def mixed_text(pats, n, seed):
    """Text with the patterns planted in random case, every byte value, and the capitals 0x41-0x5A next to their
    high-half twins 0xC1-0xDA."""
    from pfac_synth import synth_text
    t = synth_text(seed, seed + 7, n, patterns=fold(pats))
    t = random_case(t, seed + 1)
    t[:256] = np.arange(256, dtype=np.uint8)
    k = np.arange(0x41, 0x5B, dtype=np.uint8)
    t[300:352] = np.stack([k, k + 0x80], axis=1).reshape(-1)
    return t


def ref(pats, text):
    """The definition: the oracle's scan of fold(text) with the tables of fold(pats)."""
    return Oracle(fold(pats), 1, 256).scan(fold(np.ascontiguousarray(text, dtype=np.uint8)))


def test_every_entry_point_against_the_folded_reference(tmp_path):
    torch = torch_cuda()
    pats = mixed_set(3)
    tables = pf.Tables.from_bytes(pats, 1, 256, caseless=True)
    assert tables.caseless
    text = mixed_text(pats, 3 * 65536 + 4321, 3)
    o = Oracle(fold(pats), 1, 256)
    m = pf.Matcher(tables, device=0, n_streams=3, chunk_bytes=65536)
    cs = pf.Matcher(pf.Tables.from_bytes(fold(pats), 1, 256), device=0, n_streams=3, chunk_bytes=65536)
    d = torch.from_numpy(text).cuda()
    keep = d.clone()
    n = len(text)
    # scan_device: pointer offsets 0-15
    for off in range(16):
        got = m.scan_device(d, offset=off)
        same(got, o.scan(fold(text[off:])), ("offset", off))
        assert m.last_info()["launches"] == 4   # fold + detector + dense-match + ordering pass
        cs.scan_device(d, offset=off)
        assert cs.last_info()["launches"] == 3
    # n_starts < n_valid, base_pos != 0
    pos, ids = o.scan(fold(text))
    for ns in (n - 1, n // 2, 12345):
        keep_r = (pos < ns)
        same(m.scan_device(d, n_starts=ns, n_valid=n), (pos[keep_r], ids[keep_r]), ("n_starts", ns))
    same(m.scan_device(d, base_pos=7 << 20), (pos, ids), "base_pos")
    # capacity overflow and retry
    same(m.scan_device(d, cap=1), (pos, ids), "cap")
    assert len(pos) > 1
    # host pipeline over several chunks, in place on the library's stage buffers
    same(m.scan_host(text), (pos, ids), "host")
    same(m.scan_host(text, cap=3), (pos, ids), "host cap")
    # batch: per-document results, straddling matches dropped
    cuts = np.unique(np.concatenate([[0, n], np.random.default_rng(5).integers(0, n, 300)]))
    first, rec = m.scan_batch(d, cuts)
    for i in range(len(cuts) - 1):
        a, b = int(cuts[i]), int(cuts[i + 1])
        same(rec[int(first[i]):int(first[i + 1])], o.scan(fold(text[a:b])), ("doc", i))
    first2, rec2 = m.scan_batch(d, cuts, cap=2, offset=0)
    assert np.array_equal(first, first2) and np.array_equal(rec, rec2)
    # the caller's bytes are never written
    torch.cuda.synchronize()
    assert torch.equal(d, keep)
    assert np.array_equal(d.cpu().numpy(), text)
    # Job.run / run_file: absolute positions over all segments
    job = pf.Job(tables, devices=[0], streams_per_gpu=2, chunk_bytes=65536)
    for total, segs in (job.run(text), job.run_file(_write(tmp_path / "in.bin", text), n)):
        gp = np.concatenate([s[1][:, 0].astype(np.int64) + s[0] for s in segs]) if segs else np.zeros(0, np.int64)
        gi = np.concatenate([s[1][:, 1].astype(np.int64) for s in segs]) if segs else np.zeros(0, np.int64)
        assert total == len(pos) and np.array_equal(gp, pos) and np.array_equal(gi, ids)
    job.close()
    m.close()
    cs.close()


def _write(path, arr):
    path.write_bytes(np.ascontiguousarray(arr).tobytes())
    return path


def test_flows_fold_across_seams_and_commit():
    """A mixed-case match across a chunk seam is found (the carried tail is stored folded and folded again
    harmlessly); a call that overflows its capacity commits nothing, so the retry is exact."""
    torch_cuda()
    pats = random_case(b"Set-Cookie: SessionID\nHTTP/1.1 200 OK\nxYz\n", 1)
    m = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256, caseless=True), device=0)
    o = Oracle(fold(pats), 1, 256)
    rng = np.random.default_rng(2)
    streams = [random_case(b"..HTTP/1.1 200 ok..set-cookie: SESSIONid..xyZXYZ" * 40 + bytes(range(256)), s) for s in range(6)]
    fl = m.flows(len(streams))
    pos_at = [0] * len(streams)
    got = [[] for _ in streams]
    while any(pos_at[i] < len(streams[i]) for i in range(len(streams))):
        ids = [i for i in range(len(streams)) if pos_at[i] < len(streams[i])]
        chunks = []
        for i in ids:
            k = int(rng.integers(1, 40))
            chunks.append(streams[i][pos_at[i]:pos_at[i] + k])
            pos_at[i] += len(chunks[-1])
        for i, r in zip(ids, fl.feed(ids, chunks)):
            got[i].append(r)
    for i, s in enumerate(streams):
        r = np.concatenate(got[i])
        r = r[np.lexsort((r["id"], r["pos"]))]
        wp, wi = o.scan(np.frombuffer(fold(s), dtype=np.uint8))
        order = np.lexsort((wi, wp))
        assert np.array_equal(r["pos"].astype(np.int64), wp[order]) and np.array_equal(r["id"].astype(np.int64), wi[order]), i
    # commit rule: an overflowing call (cap = 1) leaves the flows unchanged; the retry inside scan() is exact
    fl2 = m.flows(2)
    a, b = random_case(b"set-cookie: sess", 9), random_case(b"ionid xyz HTTP/1.1 200 ok", 10)
    fl2.feed([0], [a])
    first, base, rec = fl2.scan([0, 1], np.frombuffer(b + b + a, dtype=np.uint8),
                                [0, len(b), len(b) + len(b + a)], cap=1)
    assert fl2.position(0) == len(a) + len(b)
    wp, wi = o.scan(np.frombuffer(fold(a + b), dtype=np.uint8))
    r0 = rec[int(first[0]):int(first[1])]
    assert sorted(zip((r0["pos"] + base[0]).tolist(), r0["id"].tolist())) == sorted(zip(wp.tolist(), wi.tolist()))
    fl.close()
    fl2.close()
    m.close()


@pytest.mark.parametrize("name", CASELESS_CASES)
def test_detector_paths_caseless(name, monkeypatch):
    """Every detector path of tests/test_detector_paths_host.py with its patterns and plants in random case: the
    case's signature (derived info, launches + 1 for the fold), device scans at pointer offsets, n_starts < n_valid,
    base_pos for the 900-byte set, and the host pipeline."""
    torch = torch_cuda()
    case = caseless_case(name)
    set_env(monkeypatch, case.spec)
    m = pf.Matcher(case.tables, device=0, n_streams=2, chunk_bytes=16384)
    check_signature(m, case)
    text, info = phase_text(case)
    rc = random_case(text, 77)
    assert np.array_equal(fold(rc), fold(text))
    expect = Expect(case, fold(rc))
    assert len(expect.pos) > len(info["plants"]) // 2
    n = len(rc)
    d = torch.from_numpy(rc).cuda()
    for off in (0, 1, 3, 8, 15):
        got = m.scan_device(d, n_starts=n - off, n_valid=n - off, offset=off)
        assert m.last_info()["launches"] == case.spec["launches"] + 1, name
        same(got, expect(off, n - off), (name, "offset", off))
    plant = info["plants"][len(info["plants"]) // 3]
    for ns in (n - 1, plant, plant + 1):
        same(m.scan_device(d, n_starts=ns, n_valid=n), expect(0, n, ns), (name, "n_starts", ns))
    if case.max_len > 513:
        a = 5000
        got = m.scan_device(d, n_starts=n - a, n_valid=n - a, base_pos=a, offset=a)
        keep = expect.pos >= a
        same(got, (expect.pos[keep] - a, expect.ids[keep]), (name, "base_pos"))
    same(m.scan_host(rc), (expect.pos, expect.ids), (name, "host"))
    assert np.array_equal(d.cpu().numpy(), rc)
    m.close()


def test_two_streams_one_context():
    """Asynchronous pfac_scan_device calls alternating between two streams of one caseless context: each is ordered
    after the previous one, which read the same folded copy."""
    torch = torch_cuda()
    import ctypes as C
    pats = mixed_set(4)
    m = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256, caseless=True), device=0)
    texts = [mixed_text(pats, 200000 + 4099 * k, 10 + k) for k in range(6)]
    wants = [ref(pats, t) for t in texts]
    s = [torch.cuda.Stream(), torch.cuda.Stream()]
    ds = [torch.from_numpy(t).cuda() for t in texts]
    outs = [torch.empty((len(w[0]) + 16, 2), dtype=torch.int32, device="cuda") for w in wants]
    cnts = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in texts]
    torch.cuda.synchronize()
    for k, d in enumerate(ds):
        off = k % 3
        m.scan_device_raw(d.data_ptr() + off, d.numel() - off, d.numel() - off, 0, outs[k].data_ptr(), outs[k].shape[0],
                          cnts[k].data_ptr(), C.c_void_p(s[k % 2].cuda_stream))
    torch.cuda.synchronize()
    for k, t in enumerate(texts):
        off = k % 3
        want = ref(pats, t[off:])
        c = int(cnts[k].item())
        assert c == len(want[0]), k
        got = outs[k][:c].cpu().numpy().astype(np.int64)
        assert np.array_equal(got[:, 0], want[0]) and np.array_equal(got[:, 1], want[1]), k
        assert np.array_equal(ds[k].cpu().numpy(), t)
    m.close()


def test_cli_caseless_with_table_cache(tmp_path):
    """GPHF_CASELESS=1 (with GPHF_TABLE_CACHE: the first run writes a PFACTBL3 cache, the second loads it, a
    case-sensitive run rebuilds): GPU_match_result.txt is the oracle's rendering of the folded scan."""
    from test_scan_gpu import render_result
    pats = mixed_set(6)
    text = mixed_text(pats, 300000, 6)
    pat, inp, cache = tmp_path / "pats", tmp_path / "in", tmp_path / "tables.cache"
    pat.write_bytes(pats)
    inp.write_bytes(text.tobytes())
    pos, ids = ref(pats, text[:-1])   # the CLI scans file size - 1 bytes (main.cc:138)
    want = render_result(pos, ids)
    for run in range(2):
        r = subprocess.run([GPHF, str(pat), "2", "256", str(inp)], cwd=tmp_path, capture_output=True, text=True,
                           env=dict(os.environ, GPHF_CASELESS="1", GPHF_TABLE_CACHE=str(cache)))
        assert r.returncode == 0, r.stderr
        assert "rebuilding" not in r.stderr
        assert cache.read_bytes()[:8] == b"PFACTBL3"
        assert (tmp_path / "GPU_match_result.txt").read_bytes() == want, run
    r = subprocess.run([GPHF, str(pat), "2", "256", str(inp)], cwd=tmp_path, capture_output=True, text=True,
                       env=dict(os.environ, GPHF_TABLE_CACHE=str(cache)))
    assert r.returncode == 0 and "rebuilding" in r.stderr
    cpos, cids = Oracle(pats, 1, 256).scan(text[:-1])
    assert (tmp_path / "GPU_match_result.txt").read_bytes() == render_result(cpos, cids)
    assert cache.read_bytes()[:8] == b"PFACTBL2"


def test_one_call_at_the_4gib_limit():
    """One device scan of the largest input a call takes, background bytes with mixed-case plants across 2^31 and at
    the last start: the fold covers every byte (64-bit indices), records equal the sparse reference."""
    torch = torch_cuda()
    from test_large_inputs_host import max_call_bytes
    case = caseless_case("A")
    n = max_call_bytes(0)
    plants = [(1 << 31) - 3, (1 << 31) + TILE - 1, 12345]
    p = max(case.lines[:50], key=len)
    last = case.lines[0]
    d = torch.full((n,), BG, dtype=torch.uint8, device="cuda")
    layout = [(at, random_case(p, at)) for at in plants] + [(n - len(last), random_case(last, 1))]
    for at, q in layout:
        d[at:at + len(q)] = torch.from_numpy(np.frombuffer(q, dtype=np.uint8).copy()).cuda()
    m = pf.Matcher(case.tables, device=0)
    got = m.scan_device(d, cap=1 << 16)
    o = Oracle(case.blob, 1, 256)
    wp, wi = [], []
    for at, q in sorted(layout):
        pos, ids = o.scan(np.frombuffer(fold(q), dtype=np.uint8))
        wp.append(pos + at)
        wi.append(ids)
    same(got, (np.concatenate(wp), np.concatenate(wi)), "4 GiB")
    for at, q in layout:   # the caller's bytes are unchanged
        assert d[at:at + len(q)].cpu().numpy().tobytes() == q
    del d
    m.close()
    torch.cuda.empty_cache()
