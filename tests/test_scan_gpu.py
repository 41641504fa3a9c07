"""Parity of the CUDA path (through the C ABI) with the oracle -- bit-exact (integer/index work).
Runs on the GPU box only; nothing here reads /root/reference."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

import phfpfac_b200 as pf
import pfac_synth as synth
from _oracle import Oracle, render_result

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GPHF = os.path.join(ROOT, "phfpfac_b200", "_build", "gphf")
ORACLE_GPHF = os.path.join(ROOT, "oracle", "_build", "oracle_gphf")


def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def check_both_paths(pats, data, width=256, n_streams=3, chunk_bytes=65536, oracle_parts=4, oracle_width=None):
    """device-resident scan and host pipeline == oracle (reference flow: 4 partitions)."""
    torch = torch_cuda()
    buf = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    o = Oracle(pats, n_parts=min(oracle_parts, pats.count(b"\n")), width=oracle_width or width)
    pos, ids = o.scan(buf)
    t = pf.Tables.from_bytes(pats, n_parts=1, width=width)
    m = pf.Matcher(t, device=0, n_streams=n_streams, chunk_bytes=chunk_bytes)
    got_h = m.scan_host(buf)
    d = torch.from_numpy(buf.copy()).cuda() if len(buf) else torch.zeros(16, dtype=torch.uint8, device="cuda")
    got_d = m.scan_device(d, n_starts=len(buf), n_valid=len(buf))
    for name, got in (("host", got_h), ("device", got_d)):
        assert len(got) == len(pos), (name, len(got), len(pos))
        assert np.array_equal(got["pos"].astype(np.int64), pos), name
        assert np.array_equal(got["id"].astype(np.int32), ids), name
    m.close()
    return pos, ids, got_d


@pytest.mark.parametrize("rname,pname,width", [
    ("experimentpattern_x_experimentinput", "experimentpattern", 256),
    ("experimentpattern_x_1M", "experimentpattern", 256),      # BASELINE.json configs[0]
    ("dictionary_x_1M", "dictionary", 256),
    ("dictionary_x_1M_single_w4096", "dictionary", 4096),
    ("dictionary_x_1M_8parts_w64", "dictionary", 64),
    ("xaa_x_1M_first64k", "xaa", 4096),
])
def test_golden_result_files(fixtures, golden, rname, pname, width):
    """Byte-identical GPU_match_result.txt images for the reference's shipped fixtures."""
    g = golden["results"][rname]
    data = {"experimentpattern_x_experimentinput": fixtures["experimentinput"][:-1],
            "xaa_x_1M_first64k": fixtures["1M"][:65536]}.get(rname, fixtures["1M"][:-1])
    pos, ids, got = check_both_paths(fixtures[pname], data, width=width)
    text = pf.format_records(got)
    assert len(got) == g["lines"] and hashlib.md5(text).hexdigest() == g["md5"]
    if "text" in g:
        assert text.decode() == g["text"]


@pytest.mark.parametrize("seed", range(10))
def test_random_patterns_and_texts(seed):
    rng = np.random.default_rng(1000 + seed)
    alpha = [2, 3, 4, 8, 26, 64, 200, 256, 5, 2][seed]
    n_pat = int(rng.integers(1, 2000))
    max_len = int(rng.integers(1, [6, 12, 40, 100, 20, 64, 16, 30, 300, 700][seed]))
    pats = set()
    usable = alpha - (1 if alpha > 10 else 0)          # byte 10 ('\n') cannot be inside a pattern
    possible = sum(usable ** L for L in range(1, min(max_len, 8) + 1))
    for _ in range(50 * n_pat):
        if len(pats) >= min(n_pat, possible):
            break
        L = int(rng.integers(1, max_len + 1))
        p = bytes(rng.integers(0, alpha, L).astype(np.uint8))
        if b"\n" not in p:
            pats.add(p)
    blob = b"".join(p + b"\n" for p in pats)
    n = int(rng.integers(1, 400000))
    text = rng.integers(0, alpha, n).astype(np.uint8)
    check_both_paths(blob, text, width=int(2 ** rng.integers(4, 13)), n_streams=int(rng.integers(1, 5)),
                     chunk_bytes=int(rng.integers(1, 8)) * 16384)


def detector_set(kind, monkeypatch):
    """-> (tables, reference scan, text) of one of the detector cases of test_detector_paths_host.py ("A": mode 0,
    "H": global mode, "J1": mode 1), with its environment set."""
    from test_detector_paths_host import get_case, phase_text, set_env
    case = get_case(kind)
    set_env(monkeypatch, case.spec)
    text, _ = phase_text(case)
    return case.tables, case.reference, text[:600000].copy()


def check_edge_sizes_and_alignment(t, ref, base, want_matches):
    torch = torch_cuda()
    m = pf.Matcher(t, device=0, n_streams=2, chunk_bytes=16384)
    d = torch.from_numpy(base.copy()).cuda()
    assert len(m.scan_host(np.zeros(0, dtype=np.uint8))) == 0
    for n in (0, 1, 2, 3, 4, 15, 16, 17, 31, 33, 4095, 4096, 4097, 16383, 16384, 16385, 32768, 49151, 65536, 70001):
        pos, ids = ref(base[:n])
        got = m.scan_host(base[:n])
        assert np.array_equal(got["pos"], pos) and np.array_equal(got["id"], ids), n
    for off in range(0, 19):
        n = 40000
        pos, ids = ref(base[off:off + n])
        got = m.scan_device(d, n_starts=n, n_valid=n, offset=off)
        assert np.array_equal(got["pos"], pos) and np.array_equal(got["id"], ids), off
        assert len(pos) > 0 or not want_matches
    m.close()


def test_edge_sizes_and_alignment():
    """Empty input, inputs shorter than a pattern, every misalignment of the device pointer,
    tile-edge lengths."""
    pats = b"abcab\nab\nb\ncabcabcabc\nabcabcabcabcabcabcabcabcabcabcabcab\n"
    o = Oracle(pats, 1, 256)
    t = pf.Tables.from_bytes(pats, 1, 256)
    base = np.frombuffer((b"abc" * 30000)[:70001], dtype=np.uint8)
    check_edge_sizes_and_alignment(t, o.scan, base, False)


@pytest.mark.parametrize("kind", ["A", "H", "J1"])
def test_edge_sizes_and_alignment_detector_sets(kind, monkeypatch):
    """The same on sets that run a detector kernel (the set above has a pattern of <= 3 bytes: the
    dense-match kernel alone): mode 0, global mode, mode 1."""
    t, ref, text = detector_set(kind, monkeypatch)
    check_edge_sizes_and_alignment(t, ref, text[8192 - 300:8192 - 300 + 70001], True)


def check_halo_semantics_and_shard_concatenation(t, ref, data, b_cut):
    """b_cut: an input length that cuts a match (reported only with the halo)."""
    torch = torch_cuda()
    pos, ids = ref(data)
    assert len(pos) > 0
    m = pf.Matcher(t, device=0)
    d = torch.from_numpy(data.copy()).cuda()
    for cuts in ([0, 1, 500000], [0, 65536, 131072 + 7, 400001, 500000], [0, 499999, 500000]):
        ps, is_ = [], []
        for a, b in zip(cuts[:-1], cuts[1:]):
            nv = min(b - a + t.max_pat_len - 1, len(data) - a)
            got = m.scan_device(d, n_starts=b - a, n_valid=nv, offset=a)
            ps.append(got["pos"].astype(np.int64) + a)
            is_.append(got["id"].astype(np.int32))
        assert np.array_equal(np.concatenate(ps), pos) and np.array_equal(np.concatenate(is_), ids), cuts
    # without the halo, a match that would straddle the end is NOT reported (walk stops at n_valid)
    got = m.scan_device(d, n_starts=b_cut, n_valid=b_cut, offset=0)
    p2, i2 = ref(data[:b_cut])
    assert np.array_equal(got["pos"], p2) and np.array_equal(got["id"], i2)
    m.close()


def test_halo_semantics_and_shard_concatenation(fixtures):
    """n_starts < n_valid: only matches STARTING in [0, n_starts) are reported, walks may read the
    halo; concatenating shards reproduces the whole scan (SURVEY.md 8(e))."""
    pats = fixtures["xab"] + b"England were\ncricket than England in the past four years.\n"
    data = np.frombuffer(fixtures["1M"][:-1], dtype=np.uint8)[:500000]
    o = Oracle(pats, 1, 256)
    t = pf.Tables.from_bytes(pats, 1, 256)
    check_halo_semantics_and_shard_concatenation(t, o.scan, data, 402 * 3 + 5)   # "England were" starts at multiples of 402


@pytest.mark.parametrize("kind", ["A", "H", "J1"])
def test_halo_semantics_and_shard_concatenation_detector_sets(kind, monkeypatch):
    """The same on sets that run a detector kernel: mode 0, global mode, mode 1."""
    t, ref, text = detector_set(kind, monkeypatch)
    data = text[:500000]
    pos, _ = ref(data)
    check_halo_semantics_and_shard_concatenation(t, ref, data, int(pos[1]) + 1)   # the second match, cut after its first byte


def test_dense_matches_and_capacity_overflow():
    """Every position matches several patterns (the reference's experimentpattern shape): record
    buffers overflow -> PFAC_ERR_OUTPUT_FULL with the required count, never a silent truncation."""
    torch = torch_cuda()
    pats = b"aaaa\naa\na\naaa\n"
    n = 300000
    data = np.full(n, ord("a"), dtype=np.uint8)
    data[::1000] = ord("b")
    o = Oracle(pats, 4, 256)
    pos, ids = o.scan(data)
    t = pf.Tables.from_bytes(pats, 1, 256)
    m = pf.Matcher(t, device=0, n_streams=2, chunk_bytes=65536)
    d = torch.from_numpy(data).cuda()
    out = torch.full((1000, 2), -7, dtype=torch.int32, device="cuda")
    import ctypes as C
    cnt = C.c_uint64(0)
    rc = pf.lib.pfac_scan_device_sync(m._h, d.data_ptr(), n, n, 0, out.data_ptr(), 999, C.byref(cnt), None)
    assert rc == -8 and cnt.value == len(pos)
    o_cpu = out.cpu().numpy()
    assert (o_cpu[999] == -7).all()            # nothing written past the capacity (contents below it: unspecified)
    h_out = np.zeros(10, dtype=pf.MATCH_DTYPE)
    rc = pf.lib.pfac_scan_host(m._h, data.ctypes.data, n, n, 0, h_out.ctypes.data, 10, C.byref(cnt))
    assert rc == -8 and cnt.value == len(pos)
    got = m.scan_host(data)                     # the wrapper retries with the reported size
    assert np.array_equal(got["pos"], pos) and np.array_equal(got["id"], ids)
    got = m.scan_device(d)
    assert np.array_equal(got["pos"], pos) and np.array_equal(got["id"], ids)
    m.close()


@pytest.mark.parametrize("n_plants", [1, 31, 32, 33, 40, 200, 3000])
def test_candidate_list_boundaries(n_plants):
    """The detector hands a tile's surviving starts to the emit kernel as a list of at most 32
    candidates; beyond that (or when a slice has too many stage-1 survivors) whole slices are handed
    over.  Plant 1..3000 matches from 300 bytes before byte 32,768 on: across that border between two tiles
    (of 8,192 starts each) and through the tiles after it."""
    torch = torch_cuda()
    pats = synth.synth_patterns(1, 3000, 3, 4, 64)
    lines = pats.split(b"\n")[:-1]
    n = 100000
    rng = np.random.default_rng(n_plants)
    text = rng.integers(0, 256, n).astype(np.uint8)
    text[text == 10] = 11
    base = 16384 * 2 - 300          # straddles the border of tiles 1 and 2
    at = base
    for i in range(n_plants):
        p = lines[int(rng.integers(0, len(lines)))]
        if at + len(p) + 2 >= n:
            break
        text[at:at + len(p)] = np.frombuffer(p, dtype=np.uint8)
        at += len(p) + int(rng.integers(0, 3))
    check_both_paths(pats, text, n_streams=2, chunk_bytes=65536, oracle_parts=4)


@pytest.mark.parametrize("min_len", [1, 4])
@pytest.mark.parametrize("spacing", [0, 37, 700])
def test_nested_patterns_many_matches_per_start(spacing, min_len):
    """One start position reporting 1..12 nested patterns (a, ab, abc, ...): the emit kernel keeps
    the first few final states of a walk in registers and walks again only past that; both ways,
    in single-candidate tiles (sparse), sorted candidate lists and whole-slice mode (dense)."""
    word = b"qwertyuiopas"
    pats = b"".join(word[:k] + b"\n" for k in range(min_len, len(word) + 1)) + b"zzzzzz\nwerty\n"
    rng = np.random.default_rng(spacing)
    chunks = []
    for i in range(3000 if spacing else 20000):
        chunks.append(word[:int(rng.integers(min_len, len(word) + 1))])
        chunks.append(b"." * spacing)
    text = np.frombuffer(b"".join(chunks), dtype=np.uint8)
    pos, ids, _ = check_both_paths(pats, text, n_streams=2, chunk_bytes=1 << 20, oracle_parts=1)
    assert len(pos) > 3 * len(chunks) // 2


def test_tables_from_reference_arrays_and_determinism(fixtures):
    """Tables handed over as canonical arrays (the thread_data fields of main.cc:19-32, here the
    oracle's) give the same records as tables built by the library, run after run."""
    torch = torch_cuda()
    o = Oracle(fixtures["dictionary"], n_parts=1, width=256)
    p = o.part(0)
    t = pf.Tables.from_arrays(p.s0, p.r, p.HT, p.val, 256, p.state_num, p.n_final, p.idmap, o.max_pat_len)
    data = np.frombuffer(fixtures["1M"][:-1], dtype=np.uint8)
    pos, ids = o.scan(data)
    m = pf.Matcher(t, device=0, n_streams=3, chunk_bytes=1 << 18)
    d = torch.from_numpy(data.copy()).cuda()
    first = m.scan_device(d)
    assert np.array_equal(first["pos"], pos) and np.array_equal(first["id"], ids)
    for _ in range(3):
        assert np.array_equal(m.scan_device(d), first)
        assert np.array_equal(m.scan_host(data), first)
    m.close()


def test_long_patterns_reference_tile_bound():
    """Patterns longer than 513 bytes: the reference cuts a walk at its 4096-byte tile + 512-byte
    halo (master_kernel.cu:141-144); positions are global (base_pos)."""
    torch = torch_cuda()
    rng = np.random.default_rng(5)
    long1 = bytes(rng.integers(97, 100, 900).astype(np.uint8))
    long2 = long1[:600] + b"z" * 100
    pats = long1 + b"\n" + long2 + b"\n" + long1[:20] + b"\nzz\n"
    o = Oracle(pats, 1, 256)
    data = bytearray(rng.integers(97, 100, 40000).astype(np.uint8).tobytes())
    for start in (0, 100, 3500, 3596, 3597, 4096 + 3000, 8192 + 3690, 12288 - 1, 20000, 39100):
        data[start:start + 900] = long1
    data[30000:30700] = long2
    data = np.frombuffer(bytes(data[:40000]), dtype=np.uint8)
    pos, ids = o.scan(data)
    assert 0 < (ids == 1).sum() < 10           # some occurrences are cut by the tile bound, some are not
    t = pf.Tables.from_bytes(pats, 1, 256)
    m = pf.Matcher(t, device=0, n_streams=2, chunk_bytes=16384)
    got = m.scan_host(data)
    assert np.array_equal(got["pos"], pos) and np.array_equal(got["id"], ids)
    d = torch.from_numpy(data.copy()).cuda()
    got = m.scan_device(d)
    assert np.array_equal(got["pos"], pos) and np.array_equal(got["id"], ids)
    # a shard that starts mid-tile must use GLOBAL tile boundaries: base_pos = 5000
    a = 5000
    got = m.scan_device(d, n_starts=len(data) - a, n_valid=len(data) - a, base_pos=a, offset=a)
    keep = pos >= a
    assert np.array_equal(got["pos"].astype(np.int64) + a, pos[keep]) and np.array_equal(got["id"], ids[keep])
    m.close()


@pytest.mark.parametrize("kind,count,seed,lo,hi,tkind,tseed,n", [
    (0, 1000, 1, 8, 32, 0, 2, 6 << 20),        # config 2 shape
    (1, 10000, 3, 4, 64, 1, 4, 6 << 20),       # config 3 shape
    (0, 30000, 5, 8, 32, 0, 6, 3 << 20),       # config 4 shape, reduced (the oracle keeps the reference's O(R^2) sort)
])
def test_baseline_config_shapes_small(kind, count, seed, lo, hi, tkind, tseed, n):
    pats = synth.synth_patterns(kind, count, seed, lo, hi)
    text = synth.synth_text(tkind, tseed, n + 1, patterns=pats)[:n]
    # results do not depend on partition count / width (SURVEY.md 3.4): the oracle uses 8 partitions
    # at width 4096 to keep its quadratic SortRows short; the product uses one automaton at width 256
    pos, ids, got = check_both_paths(pats, text, n_streams=4, chunk_bytes=1 << 20, oracle_parts=8, oracle_width=4096)
    assert len(pos) >= n // 65536


def test_full_size_properties_config2():
    """BASELINE configs[1] at full size (256 MiB): properties that do not need the oracle on the
    whole input -- sorted unique (pos,id), every record verified against the pattern text,
    shard-invariance, and exact oracle parity on sampled 1 MiB windows."""
    torch = torch_cuda()
    n = 256 << 20
    pats = synth.synth_patterns(0, 1000, 1, 8, 32)
    lines = pats.split(b"\n")[:-1]
    text = synth.synth_text(0, 2, n + 1, patterns=pats)[:n]
    t = pf.Tables.from_bytes(pats, 1, 256)
    m = pf.Matcher(t, device=0, n_streams=4)
    d = torch.from_numpy(text).cuda()
    got = m.scan_device(d)
    assert len(got) >= n // 65536 - 8
    key = got["pos"].astype(np.int64) * (1 << 20) + got["id"]
    assert (np.diff(key) > 0).all()
    for r in got[:: max(1, len(got) // 2000)]:
        p = lines[int(r["id"]) - 1]
        assert text[int(r["pos"]):int(r["pos"]) + len(p)].tobytes() == p
    got_h = m.scan_host(text)
    assert np.array_equal(got_h, got)
    o = Oracle(pats, 1, 256)
    for w in (0, 97, 255):
        a = w << 20
        b = min(n, a + (1 << 20) + t.max_pat_len - 1)
        pos, ids = o.scan(text[a:b])
        keep = pos < (1 << 20)
        sel = (got["pos"] >= a) & (got["pos"] < a + (1 << 20))
        assert np.array_equal(got["pos"][sel].astype(np.int64) - a, pos[keep]) and np.array_equal(got["id"][sel], ids[keep])
    m.close()


def test_full_size_properties_config4_tables():
    """BASELINE configs[3] pattern set (100,000 patterns, ~1.8 M states, 22 MB of tables -- beyond the
    reference's ROW_MAX/HASHTABLE_MAX) over 64 MiB: every record verified against the pattern text,
    and completeness checked by an independent brute-force (Python set of patterns) on windows."""
    torch = torch_cuda()
    n = 64 << 20
    pats = synth.synth_patterns(0, 100000, 5, 8, 32)
    lines = pats.split(b"\n")[:-1]
    text = synth.synth_text(0, 6, n + 1, patterns=pats)[:n]
    # a few extra plants of overlapping/prefix-sharing patterns at awkward places
    for i, at in enumerate((0, 16383 - 5, 16384 * 3 - 1, n - len(lines[7]))):
        p = lines[7 * i]
        text[at:at + len(p)] = np.frombuffer(p, dtype=np.uint8)
    t = pf.Tables.from_bytes(pats, 1, 256)
    m = pf.Matcher(t, device=0, n_streams=4, chunk_bytes=8 << 20)
    d = torch.from_numpy(text).cuda()
    got = m.scan_device(d)
    got_h = m.scan_host(text)
    assert np.array_equal(got, got_h)
    key = got["pos"].astype(np.int64) * (1 << 20) + got["id"]
    assert (np.diff(key) > 0).all() and len(got) >= n // 65536
    for r in got:
        p = lines[int(r["id"]) - 1]
        assert text[int(r["pos"]):int(r["pos"]) + len(p)].tobytes() == p
    index = {p: i + 1 for i, p in enumerate(lines)}
    tb = text.tobytes()
    for a in (0, 16384 * 2 - 40, (n >> 1) + 12345, n - 40000):
        b = min(n, a + 40000)
        want = []
        for i in range(a, b):
            for L in range(8, 33):
                if i + L <= n:
                    pid = index.get(tb[i:i + L])
                    if pid:
                        want.append((i, pid))
        sel = (got["pos"] >= a) & (got["pos"] < b)
        assert [(int(x["pos"]), int(x["id"])) for x in got[sel]] == want
    m.close()


def test_job_all_gpus_and_segments():
    """pfac_job over every visible GPU: segments concatenate to the oracle's list."""
    torch = torch_cuda()
    pats = synth.synth_patterns(1, 2000, 3, 4, 64)
    n = 5 * (1 << 20) + 12345
    text = synth.synth_text(1, 4, n, patterns=pats)
    o = Oracle(pats, 1, 256)
    pos, ids = o.scan(text)
    t = pf.Tables.from_bytes(pats, 1, 256)
    for devices in ([0], list(range(torch.cuda.device_count())), [0, 0, 0]):
        job = pf.Job(t, devices=devices, streams_per_gpu=2, chunk_bytes=1 << 20)
        for _ in range(2):
            total, segs = job.run(text)
            gp = np.concatenate([s[1][:, 0].astype(np.int64) + s[0] for s in segs])
            gi = np.concatenate([s[1][:, 1].astype(np.int32) for s in segs])
            assert total == len(pos) and np.array_equal(gp, pos) and np.array_equal(gi, ids)
        job.close()


def test_job_multi_segment_64bit_positions():
    """A shard larger than one 1 GiB segment: records carry 32-bit positions relative to a 64-bit
    segment base (the reference's int positions stop at 2 GiB, main.cc:79).  Properties: globally
    sorted, every record re-verified against its pattern, a match planted across the segment
    border is found, and the rendered lines carry positions > 2^30.  Positions at and above 2^31 and segment bases up
    to 4 GiB: test_job_past_4_GiB in test_large_inputs_gpu.py."""
    torch = torch_cuda()
    pats = synth.synth_patterns(0, 1000, 1, 8, 32)
    lines = pats.split(b"\n")[:-1]
    n = (1 << 30) + (3 << 20) + 17
    text = synth.synth_text(0, 2, n, patterns=pats)
    border = 1 << 30
    p0 = lines[5]
    text[border - 3:border - 3 + len(p0)] = np.frombuffer(p0, dtype=np.uint8)      # straddles the segment border
    text[n - len(lines[9]):n] = np.frombuffer(lines[9], dtype=np.uint8)            # ends exactly at input_size
    t = pf.Tables.from_bytes(pats, 1, 256)
    job = pf.Job(t, devices=[0], streams_per_gpu=4)
    total, segs = job.run(text)
    assert len(segs) == 2 and segs[1][0] == border
    gp = np.concatenate([s[1][:, 0].astype(np.int64) + s[0] for s in segs])
    gi = np.concatenate([s[1][:, 1].astype(np.int64) for s in segs])
    assert total == len(gp) >= n // 65536
    assert (np.diff(gp * 4096 + gi) > 0).all()
    assert (border - 3) in gp and (n - len(lines[9])) in gp
    for k in range(0, len(gp), max(1, len(gp) // 3000)):
        pat = lines[int(gi[k]) - 1]
        assert text[int(gp[k]):int(gp[k]) + len(pat)].tobytes() == pat
    tail = pf.format_records(np.array([(int(gp[-1] - segs[1][0]), int(gi[-1]))], dtype=pf.MATCH_DTYPE), base_pos=segs[1][0])
    assert tail == b"At position %4d, match pattern %d\n" % (int(gp[-1]), int(gi[-1]))
    job.close()


def test_shallow_ring(monkeypatch):
    """The shallowest input ring the slot scheme allows (one 8 KiB stage per slot the consumer warps can hold) instead
    of all that fits: the scheme (warps taking slots from a counter, sentinel + kend at the end) must
    not depend on the depth."""
    torch = torch_cuda()
    monkeypatch.setenv("PFAC_RING_STAGES", "1")
    pats = synth.synth_patterns(1, 3000, 3, 4, 64)
    t = pf.Tables.from_bytes(pats, 1, 256)
    m = pf.Matcher(t)
    shallow = m.derived_info()["ring_stages"]
    text = synth.synth_text(1, 9, 3 << 20, patterns=pats)
    got = m.scan_host(text)
    m.close()
    monkeypatch.delenv("PFAC_RING_STAGES")
    m2 = pf.Matcher(t)
    assert m2.derived_info()["ring_stages"] > shallow >= 4
    want = m2.scan_host(text)
    m2.close()
    assert len(want) > 0 and np.array_equal(got, want)
    o = Oracle(pats, 1, 256)
    pos, ids = o.scan(np.frombuffer(text, dtype=np.uint8)[:1 << 20])
    k = int((want["pos"] < (1 << 20) - 64).sum())
    assert np.array_equal(want["pos"][:k].astype(np.int64), pos[:k]) and np.array_equal(want["id"][:k].astype(np.int32), ids[:k])


@pytest.mark.parametrize("toggle", ["PFAC_NO_PATDIR", "PFAC_NO_W3", "PFAC_NO_PDL"])
def test_alternative_paths_agree(monkeypatch, toggle):
    """The candidates of a tile are settled through the pattern directory (all lengths probed in parallel, exact
    compare) or by the walk; stage 1 runs with or without the third-window planes; the kernels of a scan are
    programmatic dependent launches or plain ones.  Whatever the path: the oracle's records, bit for bit --
    sparse planted matches, matches side by side in one tile (two-candidate tiles), nested patterns, a match at
    the very end of the input, back-to-back scans on one stream."""
    torch = torch_cuda()
    pats = synth.synth_patterns(1, 3000, 3, 4, 64) + b"GET /index\nGET /in\nGET /index.html HTTP/1.1\n"
    text = synth.synth_text(1, 21, 6 << 20, patterns=pats).copy()
    lines = pats.split(b"\n")[:-1]
    rng = np.random.default_rng(5)
    for k in range(400):   # pairs of matches a few bytes apart, nested ones, one ending the input
        at = int(rng.integers(0, len(text) - 400))
        for j in range(2):
            q = lines[int(rng.integers(0, len(lines)))]
            text[at:at + len(q)] = np.frombuffer(q, dtype=np.uint8)
            at += len(q) + int(rng.integers(0, 40))
    last = lines[-1]
    text[len(text) - len(last):] = np.frombuffer(last, dtype=np.uint8)
    o = Oracle(pats, 1, 256)
    pos, ids = o.scan(text)
    t = pf.Tables.from_bytes(pats, 1, 256)
    d = torch.from_numpy(text).cuda()
    got = {}
    for off in (False, True):
        if off:
            monkeypatch.setenv(toggle, "1")
        m = pf.Matcher(t, device=0, n_streams=3, chunk_bytes=1 << 20)
        for _ in range(3):   # back to back on one stream
            r = m.scan_device(d, n_starts=len(text), n_valid=len(text))
        got[off] = (r, m.scan_host(text))
        m.close()
    monkeypatch.delenv(toggle)
    for off, (rd, rh) in got.items():
        for r in (rd, rh):
            assert len(r) == len(pos) and len(pos) > 800, (toggle, off, len(r), len(pos))
            assert np.array_equal(r["pos"].astype(np.int64), pos) and np.array_equal(r["id"].astype(np.int32), ids), (toggle, off)


def test_device_scans_on_two_streams_share_one_context(fixtures):
    """pfac_scan_device calls of one context enqueued on different streams are ordered on the device
    (they share the control block and the tile directory): interleave two inputs on two streams."""
    torch = torch_cuda()
    t = pf.Tables.from_bytes(fixtures["dictionary"], 1, 256)
    m = pf.Matcher(t)
    rng = np.random.default_rng(5)
    base = np.frombuffer(fixtures["1M"], dtype=np.uint8)
    texts = [base[:700000].copy(), np.roll(base, 12345)[:400000].copy()]
    want = [m.scan_host(x) for x in texts]
    d_in = [torch.from_numpy(x).cuda() for x in texts]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = [torch.empty((len(w) + 16, 2), dtype=torch.int32, device="cuda") for w in want]
    cnts = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in want]
    torch.cuda.synchronize()
    for rep in range(6):
        i = rep & 1
        m.scan_device_raw(d_in[i].data_ptr(), len(texts[i]), len(texts[i]), 0, outs[i].data_ptr(), outs[i].shape[0],
                          cnts[i].data_ptr(), streams[i].cuda_stream)
    torch.cuda.synchronize()
    for i in range(2):
        n = int(cnts[i].item())
        assert n == len(want[i])
        got = outs[i][:n].cpu().numpy()
        assert np.array_equal(got[:, 0].astype(np.uint32), want[i]["pos"]) and np.array_equal(got[:, 1].astype(np.uint32), want[i]["id"])
    m.close()


def test_host_register_in_place(fixtures):
    """pfac_host_register: scanning from caller memory pinned in place gives the same records."""
    t = pf.Tables.from_bytes(fixtures["dictionary"], 1, 256)
    m = pf.Matcher(t)
    text = np.frombuffer(fixtures["1M"], dtype=np.uint8).copy()
    want = m.scan_host(text)
    with pf.pinned(text) as a:
        got = m.scan_host(a)
    assert np.array_equal(got, want)
    with pytest.raises(pf.PfacError) as e:
        pf.check(pf.lib.pfac_host_register(None, 0, 0))
    assert e.value.code == -5
    m.close()


def test_cli_byte_identical_result_file(fixtures, golden, tmp_path):
    """gphf <pattern file> <streams> <width> <input file> -> GPU_match_result.txt (main.cc:94,335)."""
    pat = tmp_path / "experimentpattern"
    pat.write_bytes(fixtures["experimentpattern"])
    inp = tmp_path / "1M"
    inp.write_bytes(fixtures["1M"])
    r = subprocess.run([GPHF, str(pat), "1", "256", str(inp)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = (tmp_path / "GPU_match_result.txt").read_bytes()
    g = golden["results"]["experimentpattern_x_1M"]
    assert out.count(b"\n") == g["lines"] and hashlib.md5(out).hexdigest() == g["md5"]
    # dictionary, other stream counts / widths: still the same bytes; and equal to the oracle CLI
    dic = tmp_path / "dict"
    dic.write_bytes(fixtures["dictionary"])
    for (streams, width), reader in zip(((4, 64), (2, 4096), (3, 256)), ("mmap", "fread", "stream")):
        r = subprocess.run([GPHF, str(dic), str(streams), str(width), str(inp)], cwd=tmp_path, capture_output=True,
                           text=True, env=dict(os.environ, GPHF_READER=reader, GPHF_SIDECAR=str(tmp_path / "records.pfacrec")))
        assert r.returncode == 0, r.stderr
        assert f"input reader: {reader}" in r.stdout
        out = (tmp_path / "GPU_match_result.txt").read_bytes()
        assert hashlib.md5(out).hexdigest() == golden["results"]["dictionary_x_1M"]["md5"]
        # GPHF_SIDECAR: the compact records as a binary file; the text file is a pure function of it
        spos, sid = pf.read_sidecar(tmp_path / "records.pfacrec")
        assert len(spos) == golden["results"]["dictionary_x_1M"]["lines"]
        assert hashlib.md5(render_result(spos.astype(np.int64), sid.astype(np.int64))).hexdigest() == golden["results"]["dictionary_x_1M"]["md5"]
    # GPHF_TABLE_CACHE: first run builds and writes the cache, second run loads it; same bytes out
    cache = tmp_path / "tables.cache"
    for run in range(2):
        r = subprocess.run([GPHF, str(dic), "2", "256", str(inp)], cwd=tmp_path, capture_output=True, text=True,
                           env=dict(os.environ, GPHF_TABLE_CACHE=str(cache)))
        assert r.returncode == 0 and cache.exists(), r.stderr
        out = (tmp_path / "GPU_match_result.txt").read_bytes()
        assert hashlib.md5(out).hexdigest() == golden["results"]["dictionary_x_1M"]["md5"]
    # a cache built from another width or another pattern file is not trusted: the tables are rebuilt
    r = subprocess.run([GPHF, str(dic), "2", "64", str(inp)], cwd=tmp_path, capture_output=True, text=True,
                       env=dict(os.environ, GPHF_TABLE_CACHE=str(cache)))
    assert r.returncode == 0 and "rebuilding" in r.stderr
    assert hashlib.md5((tmp_path / "GPU_match_result.txt").read_bytes()).hexdigest() == golden["results"]["dictionary_x_1M"]["md5"]
    r = subprocess.run([GPHF, str(pat), "2", "64", str(inp)], cwd=tmp_path, capture_output=True, text=True,
                       env=dict(os.environ, GPHF_TABLE_CACHE=str(cache)))
    assert r.returncode == 0 and "rebuilding" in r.stderr
    assert hashlib.md5((tmp_path / "GPU_match_result.txt").read_bytes()).hexdigest() == g["md5"]
    # usage / error behaviour (main.cc:93-96, :131-135)
    assert subprocess.run([GPHF, str(pat)], cwd=tmp_path, capture_output=True).returncode == 255
    assert subprocess.run([GPHF, str(pat), "1", "256", str(tmp_path / "nope")], cwd=tmp_path, capture_output=True).returncode == 1
    assert subprocess.run([GPHF, str(tmp_path / "nope"), "1", "256", str(inp)], cwd=tmp_path, capture_output=True).returncode == 1
    assert subprocess.run([GPHF, str(pat), "1", "100", str(inp)], cwd=tmp_path, capture_output=True).returncode == 1


def test_job_streams_a_file(tmp_path):
    """pfac_job_run_file: reader threads fill a ring of pinned 64 MiB buffers while the chunks that are in
    are scanned -- the same records as scanning the whole buffer, across chunk and segment borders."""
    torch_cuda()
    pats = synth.synth_patterns(1, 2000, 3, 4, 64)
    n = (130 << 20) + 12345                   # three chunks, the last one ragged
    text = synth.synth_text(1, 21, n, patterns=pats)
    border = 64 << 20
    text[border - 3:border + 2] = np.frombuffer(b"GET /", dtype=np.uint8)     # a match across a chunk border
    pats += b"GET /\n"
    f = tmp_path / "big.bin"
    text.tofile(f)
    t = pf.Tables.from_bytes(pats, 1, 256)
    job = pf.Job(t, devices=[0], streams_per_gpu=3)
    nm, segs = job.run(text)
    nm2, segs2 = job.run_file(str(f), n)
    assert nm == nm2 > 0
    a = np.concatenate([np.stack([r[:, 0].astype(np.int64) + b, r[:, 1].astype(np.int64)], 1) for b, r in segs if len(r)])
    b = np.concatenate([np.stack([r[:, 0].astype(np.int64) + b2, r[:, 1].astype(np.int64)], 1) for b2, r in segs2 if len(r)])
    assert np.array_equal(a, b) and (a[:, 0] == border - 3).any()
    job.close()


def test_c_host_example_end_to_end(fixtures, golden, tmp_path):
    """examples/host_c_abi.c (plain C against include/pfac_b200.h): tables, multi-GPU job, writer --
    byte-identical GPU_match_result.txt."""
    from test_abi_host import _build_c_example
    torch_cuda()
    exe = _build_c_example(tmp_path)
    pat = tmp_path / "dict"
    pat.write_bytes(fixtures["dictionary"])
    inp = tmp_path / "1M"
    inp.write_bytes(fixtures["1M"])
    r = subprocess.run([str(exe), str(pat), "256", str(inp)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, (r.stdout, r.stderr)
    out = (tmp_path / "GPU_match_result.txt").read_bytes()
    assert hashlib.md5(out).hexdigest() == golden["results"]["dictionary_x_1M"]["md5"]


def test_records_equal_the_reference_gpu_kernel(ref_live):
    """The reference's own TraceTable_kernel (master_kernel.cu built for sm_100a by `make -C oracle
    refgpu`, texture fetches replaced by __ldg): its dense result, sifted the way main.cc:304-350 does,
    equals the product's records for the config-3 pattern set -- as stored in tests/golden/ref_live.json,
    and run live on this GPU too where oracle/_ref was built."""
    import json
    from _ref_sets import gpu_kernel_case
    torch = torch_cuda()
    want = ref_live["gpu_kernel_config3"]
    pats, text = gpu_kernel_case()
    assert len(text) == want["bytes"] and len(want["pos"]) > 0
    m = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256))
    for got in (m.scan_host(text), m.scan_device(torch.from_numpy(text).cuda())):
        assert got["pos"].astype(np.int64).tolist() == want["pos"] and got["id"].astype(np.int64).tolist() == want["id"]
    m.close()
    tool = os.path.join(os.path.dirname(os.path.abspath(__file__)), "refgpu_bench.py")
    r = subprocess.run([sys.executable, tool, "--mib", "3"], capture_output=True, text=True, timeout=170)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    if "unavailable" not in line:
        assert line["records_equal_to_product"] is True and line["matches"] == len(want["pos"]), line
