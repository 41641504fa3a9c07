"""Per-pattern case rules on the B200: every scan entry point of a mixed set returns, record for record, what the
reference of tests/_case_rules_ref.py returns (the caseless lines' oracle over the folded text merged with the exact
lines' oracle over the text, by (pos, length, id)).  The text is folded out of place, the unchanged detector reports
owner ids, and the verify pass expands them against the original bytes: two more launches than the caseless set."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import phfpfac_b200 as pf
from phfpfac_b200._lib import PFAC_ERR_OUTPUT_FULL, lib
from _case_rules_ref import CaseRulesRef
from _caseless_ref import fold
from test_case_rules_host import alternating
from test_caseless_gpu import mixed_set, mixed_text
from test_caseless_host import CASELESS_CASES, caseless_case, random_case
from test_detector_paths_gpu import check_signature, same
from test_detector_paths_host import BG, brute_force, lines_of, phase_text, set_env

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GPHF = os.path.join(ROOT, "phfpfac_b200", "_build", "gphf")


def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def rules_text(pats, n, seed):
    """mixed_text (the patterns planted in random case) followed by the patterns planted in their file case, so that
    exact lines both fail and pass their check."""
    from pfac_synth import synth_text
    return np.concatenate([mixed_text(pats, n // 2, seed), synth_text(seed + 3, seed + 9, n - n // 2, patterns=pats)])


def test_every_entry_point_against_the_reference(tmp_path):
    torch = torch_cuda()
    pats = mixed_set(3)
    n_pat = pats.count(b"\n")
    rules = alternating(n_pat, 3)
    tables = pf.Tables.from_bytes(pats, 1, 256, caseless=rules)
    assert not tables.caseless and tables.case_rules.tolist() == rules.tolist()
    ref = CaseRulesRef(pats, rules)
    text = rules_text(pats, 3 * 65536 + 4321, 3)
    m = pf.Matcher(tables, device=0, n_streams=3, chunk_bytes=65536)
    d = torch.from_numpy(text).cuda()
    keep = d.clone()
    n = len(text)
    pos, ids = ref.scan(text)
    exact = rules[ids - 1] == 0
    assert exact.sum() > 20 and (~exact).sum() > 20   # both classes report
    for off in range(16):
        same(m.scan_device(d, offset=off), ref.scan(text[off:]), ("offset", off))
        assert m.last_info()["launches"] == 6   # fold + detector + dense-match + ordering pass + 2 verify
    for ns in (n - 1, n // 2, 12345):
        k = pos < ns
        same(m.scan_device(d, n_starts=ns, n_valid=n), (pos[k], ids[k]), ("n_starts", ns))
    same(m.scan_device(d, base_pos=7 << 20), (pos, ids), "base_pos")
    # host pipeline: sub-chunks of 64 KiB (pos_bias != 0), folded out of place on every stage
    same(m.scan_host(text), (pos, ids), "host")
    assert m.last_info()["chunks"] == 4
    same(m.scan_host(text, cap=3), (pos, ids), "host cap")
    # batch and docs: per-document results
    cuts = np.unique(np.concatenate([[0, n], np.random.default_rng(5).integers(0, n, 300)]))
    first, rec = m.scan_batch(d, cuts)
    for i in range(len(cuts) - 1):
        a, b = int(cuts[i]), int(cuts[i + 1])
        same(rec[int(first[i]):int(first[i + 1])], ref.scan(text[a:b]), ("doc", i))
    docs = [text[int(cuts[i]):int(cuts[i + 1])] for i in range(0, len(cuts) - 1, 7)]
    for i, r in enumerate(m.scan_docs(docs)):
        same(r, ref.scan(docs[i]), ("scan_docs", i))
    torch.cuda.synchronize()
    assert torch.equal(d, keep)
    m.close()


def _sorted_flow(recs, lens):
    r = np.concatenate(recs) if recs else np.zeros(0, pf.FLOW_MATCH_DTYPE)
    p, i = r["pos"].astype(np.int64), r["id"].astype(np.int64)
    o = np.lexsort((i, lens[i], p))
    return p[o], i[o]


def test_flows_check_exact_patterns_across_seams():
    """Exact patterns straddling chunk seams, with the case mismatch on the tail side only and on the chunk side
    only: the tails stay unfolded, so the check on the next call sees the original bytes."""
    torch_cuda()
    pats = b"Set-Cookie: SessionID\nHTTP/1.1 200 OK\nxYz\nX-Token\n"
    rules = [0, 1, 1, 0]
    m = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256, caseless=rules), device=0)
    ref = CaseRulesRef(pats, rules)
    P = b"Set-Cookie: SessionID"
    streams = [b"..%s..HTTP/1.1 200 ok..xyZ.X-Token.x-token" % P,
               b"..s" + P[1:] + b"..",            # mismatch before the seam (tail side)
               b".." + P[:-1] + b"d..",           # mismatch after the seam (chunk side)
               b".." + P + b".." + P.lower() + b"..X-Token"]
    fl = m.flows(len(streams))
    got = [[] for _ in streams]
    cut = 2 + len(P) // 2
    for i, r in zip(range(len(streams)), fl.feed(list(range(len(streams))), [s[:cut] for s in streams])):
        got[i].append(r)
    for i, r in zip(range(len(streams)), fl.feed(list(range(len(streams))), [s[cut:] for s in streams])):
        got[i].append(r)
    for i, s in enumerate(streams):
        same_pos, same_ids = _sorted_flow(got[i], ref.lens)
        wp, wi = ref.scan(np.frombuffer(s, dtype=np.uint8))
        assert np.array_equal(same_pos, wp) and np.array_equal(same_ids, wi), i
    # random chunking of random-case streams
    rng = np.random.default_rng(2)
    streams = [random_case(b"..HTTP/1.1 200 ok..%s..xyZ X-Token" % P * 30, s) + P * 3 for s in range(6)]
    fl2 = m.flows(len(streams))
    at = [0] * len(streams)
    got = [[] for _ in streams]
    while any(at[i] < len(streams[i]) for i in range(len(streams))):
        live = [i for i in range(len(streams)) if at[i] < len(streams[i])]
        chunks = []
        for i in live:
            k = int(rng.integers(1, 40))
            chunks.append(streams[i][at[i]:at[i] + k])
            at[i] += len(chunks[-1])
        for i, r in zip(live, fl2.feed(live, chunks)):
            got[i].append(r)
    for i, s in enumerate(streams):
        gp, gi = _sorted_flow(got[i], ref.lens)
        wp, wi = ref.scan(np.frombuffer(s, dtype=np.uint8))
        assert np.array_equal(gp, wp) and np.array_equal(gi, wi), i
    fl.close()
    fl2.close()
    m.close()


def test_group_of_case_variants():
    """The 8 case variants of get as exact lines, a caseless GET and a byte-equal exact duplicate: at each variant
    the live exact line of that spelling and the caseless line report, in ascending id order."""
    torch = torch_cuda()
    variants = [bytes(c - 32 if (k >> j) & 1 else c for j, c in enumerate(b"get")) for k in range(8)]
    lines = variants + [b"GET", variants[5]]       # ids 1-8 exact, 9 caseless, 10 = exact duplicate of line 6
    rules = [0] * 8 + [1, 0]
    blob = b"".join(p + b"\n" for p in lines)
    t = pf.Tables.from_bytes(blob, 1, 256, caseless=rules)
    assert t.pattern_lengths().tolist() == [0] + [3] * 5 + [0] + [3] * 4
    text = np.frombuffer(b".".join(variants) + b".", dtype=np.uint8)
    m = pf.Matcher(t, device=0)
    got = m.scan_device(torch.from_numpy(text.copy()).cuda())
    same(got, CaseRulesRef(blob, rules).scan(text), "group")
    for k, v in enumerate(variants):
        at = got["id"][got["pos"] == 4 * k].tolist()
        assert at == sorted([10 if k == 5 else k + 1, 9]), (v, at)
    same(m.scan_host(text), CaseRulesRef(blob, rules).scan(text), "group host")
    m.close()


def test_letterless_and_high_half_exact_patterns():
    """Exact lines without letters match wherever their fold does; exact lines with bytes 0xC1-0xDA (which do not
    fold) next to letters are checked byte for byte."""
    torch = torch_cuda()
    blob = b"123\n--=\n\xc1B\n\xc1b\n\xdaz\xc1\nQ\xda\nabc1\nABC1\n"
    rules = [0, 0, 0, 1, 0, 0, 1, 0]
    rng = np.random.default_rng(4)
    alpha = np.frombuffer(b"123-=\xc1\xe1\xda\xfaBbZzQqAaCc", dtype=np.uint8)
    text = alpha[rng.integers(0, len(alpha), 200000)]
    m = pf.Matcher(pf.Tables.from_bytes(blob, 1, 256, caseless=rules), device=0, n_streams=2, chunk_bytes=16384)
    ref = CaseRulesRef(blob, rules)
    d = torch.from_numpy(text.copy()).cuda()
    for off in (0, 5):
        same(m.scan_device(d, offset=off), ref.scan(text[off:]), ("offset", off))
    same(m.scan_host(text), ref.scan(text), "host")
    m.close()


def mixed_case(name):
    """A detector-path case as a mixed set: its caseless lines in random case, its exact lines as they are (the
    texts plant them so); rules drawn with a seed."""
    case = caseless_case(name)
    rules = alternating(len(case.lines), len(name))
    file_lines = [random_case(p, 7 + i) if r else p for i, (p, r) in enumerate(zip(case.lines, rules))]
    blob = b"".join(p + b"\n" for p in file_lines)
    assert lines_of(blob) == file_lines
    return case, rules, blob


def mixed_reference(case, rules, blob, text):
    if case.spec.get("ref") == "brute":   # (large sets: no oracle) the two rule classes, brute force, merged
        lines = lines_of(blob)
        pos, ids = [], []
        for cls in (1, 0):
            sel = [i for i in range(len(lines)) if rules[i] == cls]
            if sel:
                p, i = brute_force([fold(lines[k]) if cls else lines[k] for k in sel], fold(text) if cls else text)
                pos.append(p)
                ids.append(np.array(sel, dtype=np.int64)[i.astype(np.int64) - 1] + 1)
        pos, ids = np.concatenate(pos), np.concatenate(ids)
        lens = np.array([0] + [len(p) for p in lines], dtype=np.int64)
        o = np.lexsort((ids, lens[ids], pos))
        return pos[o], ids[o]
    return CaseRulesRef(blob, rules).scan(text)


@pytest.mark.parametrize("name", CASELESS_CASES)
def test_detector_paths_mixed(name, monkeypatch):
    """Every detector path with mixed rules: the case's signature (launches = the caseless launches + the verify
    pass), device scans at pointer offsets over the planted text and its random-case copy, n_starts < n_valid,
    base_pos for the 900-byte set, and the host pipeline."""
    torch = torch_cuda()
    case, rules, blob = mixed_case(name)
    set_env(monkeypatch, case.spec)
    t = pf.Tables.from_bytes(blob, 1, 256, caseless=rules)
    m = pf.Matcher(t, device=0, n_streams=2, chunk_bytes=16384)
    check_signature(m, case)
    text, info = phase_text(case)
    for tx in (text, random_case(text, 77)):
        n = len(tx)
        full = mixed_reference(case, rules, blob, tx)
        assert len(full[0]) > 0
        d = torch.from_numpy(tx.copy()).cuda()
        for off in (0, 1, 3, 8, 15):
            got = m.scan_device(d, n_starts=n - off, n_valid=n - off, offset=off)
            assert m.last_info()["launches"] == case.spec["launches"] + 3, name
            if case.max_len > 513:
                want = mixed_reference(case, rules, blob, tx[off:])
            else:
                k = full[0] >= off
                want = (full[0][k] - off, full[1][k])
            same(got, want, (name, "offset", off))
        plant = info["plants"][len(info["plants"]) // 3]
        if case.max_len <= 513:
            for ns in (n - 1, plant, plant + 1):
                k = full[0] < ns
                same(m.scan_device(d, n_starts=ns, n_valid=n), (full[0][k], full[1][k]), (name, "n_starts", ns))
        else:
            a = 5000
            got = m.scan_device(d, n_starts=n - a, n_valid=n - a, base_pos=a, offset=a)
            k = full[0] >= a
            same(got, (full[0][k] - a, full[1][k]), (name, "base_pos"))
        same(m.scan_host(tx), full, (name, "host"))
        assert np.array_equal(d.cpu().numpy(), tx)
    m.close()


def _raw_scan(m, d, cap):
    import torch
    out = torch.zeros((cap + 16, 2), dtype=torch.int32, device="cuda")
    cnt = C.c_uint64(0)
    torch.cuda.synchronize()
    rc = lib.pfac_scan_device_sync(m._h, d.data_ptr(), d.numel(), d.numel(), 0, out.data_ptr(), cap, C.byref(cnt), None)
    return rc, cnt.value, out


def test_capacity_and_one_rescan():
    """cap 0, cap below the detector's own count, cap between the expanded count and that count (exact members
    that fail make the expanded count smaller): PFAC_ERR_OUTPUT_FULL, nothing past d_out[cap), and one rescan with
    the returned count gives every record.  With the detector's records inside their buffer (max(cap, 4096) records,
    held by the context once grown) the count is exact.  Each cap runs on a fresh context."""
    torch = torch_cuda()
    blob = b"abc\nXyZ\nxyz\nQQQq\n"
    rules = [1, 0, 1, 0]
    ref = CaseRulesRef(blob, rules)
    tables = pf.Tables.from_bytes(blob, 1, 256, caseless=rules)
    unit = b"abc xyz XyZ XYZ qqqq qqqq qqqq "    # 7 detector records, 5 expanded
    for reps, caps in ((400, (0, 1999)), (2000, (0, 5000, 12000))):
        text = np.frombuffer(unit * reps, dtype=np.uint8)
        want = ref.scan(text)
        assert len(want[0]) == 5 * reps
        d = torch.from_numpy(text.copy()).cuda()
        for cap in caps:
            m = pf.Matcher(tables, device=0)
            rc, cnt, out = _raw_scan(m, d, cap)
            assert rc == PFAC_ERR_OUTPUT_FULL, (reps, cap, rc)
            if 7 * reps <= max(cap, 4096):
                assert cnt == 5 * reps
            else:
                assert cnt == 7 * reps * 2   # the detector's count x the largest group
            assert out[cap:].abs().sum().item() == 0   # nothing past d_out[cap)
            rc, cnt2, out = _raw_scan(m, d, cnt)
            assert rc == 0 and cnt2 == 5 * reps
            got = out[:cnt2].cpu().numpy().astype(np.int64)
            assert np.array_equal(got[:, 0], want[0]) and np.array_equal(got[:, 1], want[1]), (reps, cap)
            m.close()
    # flows: a call that overflows commits nothing
    m = pf.Matcher(tables, device=0)
    fl = m.flows(2)
    vals = torch.from_numpy(np.frombuffer(unit * 50, dtype=np.uint8).copy()).cuda()
    offs = np.array([0, 100, len(unit) * 50], dtype=np.uint64)
    ids = np.array([0, 1], dtype=np.uint32)
    out = torch.zeros((4, 2), dtype=torch.int32, device="cuda")
    first = torch.zeros(3, dtype=torch.int64, device="cuda")
    base = np.zeros(2, dtype=np.uint64)
    cnt = C.c_uint64(0)
    torch.cuda.synchronize()
    rc = lib.pfac_scan_flows_device_sync(fl._h, vals.data_ptr(), offs.ctypes.data, ids.ctypes.data, 2, out.data_ptr(), 4,
                                         first.data_ptr(), base.ctypes.data, C.byref(cnt), None)
    assert rc == PFAC_ERR_OUTPUT_FULL and fl.position(0) == 0 and fl.position(1) == 0
    first_r, base_r, rec = fl.scan([0, 1], vals, offs)
    assert fl.position(0) == 100
    for i in range(2):
        a, b = int(offs[i]), int(offs[i + 1])
        same(rec[int(first_r[i]):int(first_r[i + 1])], ref.scan(np.frombuffer(unit * 50, dtype=np.uint8)[a:b]), ("flow", i))
    fl.close()
    m.close()


def test_batch_whose_verify_pass_overflows():
    """A mixed batch runs the verify pass and then the batch split pass over one per-CTA count buffer.  With the
    detector's records beyond their buffer (max(cap, 4096) records) the verify pass overflows first and the split
    pass passes its count on: PFAC_ERR_OUTPUT_FULL with a count of at least the exact one, nothing past d_out[cap),
    and one rescan with that count gives every document's records and doc_first.  A smaller batch and a flow call
    on the same context then match the reference: nothing carries over from one pass or call to the next."""
    torch = torch_cuda()
    blob = b"abc\nXyZ\nxyz\nQQQq\n"
    rules = [1, 0, 1, 0]
    ref = CaseRulesRef(blob, rules)
    unit = b"abc xyz XyZ XYZ qqqq qqqq qqqq "    # 7 detector records, 5 expanded
    m = pf.Matcher(pf.Tables.from_bytes(blob, 1, 256, caseless=rules), device=0)

    def per_doc(text, cuts, first, rec, what):
        want_first = [0]
        for i in range(len(cuts) - 1):
            a, b = int(cuts[i]), int(cuts[i + 1])
            wp, wi = ref.scan(text[a:b])
            got = rec[int(first[i]):int(first[i + 1])]
            assert np.array_equal(got[:, 0], wp) and np.array_equal(got[:, 1], wi), (what, i)
            want_first.append(want_first[-1] + len(wp))
        assert np.array_equal(first, want_first), what
        return want_first[-1]

    text = np.frombuffer(unit * 2000, dtype=np.uint8)
    n = len(text)
    cuts = np.unique(np.concatenate([[0, n], np.random.default_rng(8).integers(0, n, 40)])).astype(np.uint64)
    exact = sum(len(ref.scan(text[int(cuts[i]):int(cuts[i + 1])])[0]) for i in range(len(cuts) - 1))
    d = torch.from_numpy(text.copy()).cuda()

    def batch(cap):
        out = torch.zeros((cap + 16, 2), dtype=torch.int32, device="cuda")
        first = torch.zeros(len(cuts), dtype=torch.int64, device="cuda")
        cnt = C.c_uint64(0)
        torch.cuda.synchronize()
        rc = lib.pfac_scan_batch_device_sync(m._h, d.data_ptr(), cuts.ctypes.data, len(cuts) - 1, out.data_ptr(), cap,
                                             first.data_ptr(), C.byref(cnt), None)
        return rc, cnt.value, out, first

    cap = 100
    rc, cnt, out, _ = batch(cap)
    assert 7 * 2000 > max(cap, 4096)
    assert rc == PFAC_ERR_OUTPUT_FULL and cnt >= exact, (rc, cnt, exact)
    assert out[cap:].abs().sum().item() == 0   # nothing past d_out[cap)
    rc, cnt2, out, first = batch(cnt)
    assert rc == 0 and cnt2 == exact
    rec = out[:cnt2].cpu().numpy().astype(np.int64)
    assert per_doc(text, cuts, first.cpu().numpy(), rec, "rescan") == exact
    # a smaller batch on the same context
    small = np.frombuffer(unit * 300, dtype=np.uint8)
    cuts2 = np.unique(np.concatenate([[0, len(small)], np.random.default_rng(9).integers(0, len(small), 25)]))
    first2, rec2 = m.scan_batch(small, cuts2)
    rec2 = np.stack([rec2["pos"].astype(np.int64), rec2["id"].astype(np.int64)], axis=1)
    per_doc(small, cuts2, first2.astype(np.int64), rec2, "second batch")
    # and a flow call
    fl = m.flows(2)
    offs = np.array([0, 1000, len(small)], dtype=np.uint64)
    chunk_first, base, rec3 = fl.scan([0, 1], small, offs)
    assert base.tolist() == [0, 0]
    rec3 = np.stack([rec3["pos"].astype(np.int64), rec3["id"].astype(np.int64)], axis=1)
    per_doc(small, offs, chunk_first.astype(np.int64), rec3, "flows")
    fl.close()
    m.close()


def test_uniform_rules_launch_and_report_as_the_uniform_sets():
    torch = torch_cuda()
    pats = mixed_set(5)
    n_pat = pats.count(b"\n")
    text = rules_text(pats, 300000, 5)
    d = torch.from_numpy(text).cuda()
    for rule, caseless, launches in ((1, True, 4), (0, False, 3)):
        a = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256, caseless=[rule] * n_pat), device=0)
        b = pf.Matcher(pf.Tables.from_bytes(pats, 1, 256, caseless=caseless), device=0)
        ga, gb = a.scan_device(d), b.scan_device(d)
        assert a.last_info()["launches"] == b.last_info()["launches"] == launches
        assert np.array_equal(ga, gb)
        assert a.derived_info()["table_bytes"] == b.derived_info()["table_bytes"]
        a.close()
        b.close()


def test_cli_nocase_lines_with_table_cache(tmp_path):
    """GPHF_NOCASE_LINES: the first run builds and writes the cache, the second loads it, changed rules rebuild."""
    from test_scan_gpu import render_result
    pats = mixed_set(6)
    n_pat = pats.count(b"\n")
    text = rules_text(pats, 300000, 6)
    pat, inp, cache, nc = tmp_path / "pats", tmp_path / "in", tmp_path / "tables.cache", tmp_path / "nocase"
    pat.write_bytes(pats)
    inp.write_bytes(text.tobytes())
    for k, rules in enumerate((alternating(n_pat, 6), alternating(n_pat, 7))):
        nc.write_text("".join(f"{i + 1}\n" for i in np.nonzero(rules)[0]))
        pos, ids = CaseRulesRef(pats, rules).scan(text[:-1])   # the CLI scans file size - 1 bytes (main.cc:138)
        for run in range(2):
            r = subprocess.run([GPHF, str(pat), "2", "256", str(inp)], cwd=tmp_path, capture_output=True, text=True,
                               env=dict(os.environ, GPHF_NOCASE_LINES=str(nc), GPHF_TABLE_CACHE=str(cache)))
            assert r.returncode == 0, r.stderr
            assert ("rebuilding" in r.stderr) == (k == 1 and run == 0), (k, run, r.stderr)
            assert cache.read_bytes()[:8] == b"PFACTBL3"
            assert (tmp_path / "GPU_match_result.txt").read_bytes() == render_result(pos, ids), (k, run)


def test_one_call_past_2gib():
    """One device scan of 2^31 + 1 bytes with an exact plant across 2^31 (its last byte is byte 2^31), in the right
    case and then in the wrong case: the verify pass reads the original text with 64-bit indices."""
    torch = torch_cuda()
    case, rules, blob = mixed_case("A")
    lines = lines_of(blob)
    exact = max((p for p, r in zip(lines, rules) if r == 0 and any(65 <= c <= 90 or 97 <= c <= 122 for c in p)), key=len)
    n = (1 << 31) + 1
    at = n - len(exact)
    m = pf.Matcher(pf.Tables.from_bytes(blob, 1, 256, caseless=rules), device=0)
    d = torch.full((n,), BG, dtype=torch.uint8, device="cuda")
    ref = CaseRulesRef(blob, rules)
    for q in (exact, exact.swapcase()):
        d[at:at + len(q)] = torch.from_numpy(np.frombuffer(q, dtype=np.uint8).copy()).cuda()
        got = m.scan_device(d, cap=1 << 12)
        win = np.full(len(q) + 128, BG, dtype=np.uint8)
        win[64:64 + len(q)] = np.frombuffer(q, dtype=np.uint8)
        wp, wi = ref.scan(win)
        same(got, (wp - 64 + at, wi), ("2 GiB", q))
        assert (exact in [lines[i - 1] for i in wi.tolist()]) == (q == exact)
        assert d[at:at + len(q)].cpu().numpy().tobytes() == q
    del d
    m.close()
    torch.cuda.empty_cache()
