"""Per-pattern case rules (PFAC_PATTERNS_CASE_RULES) on the host: the reference, the builder's refusals, the tables,
lengths, rules, hashes and cache files of mixed sets, and the CLI's GPHF_NOCASE_LINES parsing.  The GPU side is
tests/test_case_rules_gpu.py."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

import phfpfac_b200 as pf
from phfpfac_b200._lib import PFAC_ERR_ARG, lib
from _case_rules_ref import CaseRulesRef, brute_force, patterns_of
from _caseless_ref import fold, octal_file
from test_caseless_host import random_case, same_tables

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GPHF = os.path.join(ROOT, "phfpfac_b200", "_build", "gphf")


def alternating(n, seed):
    """One rule per pattern, drawn with a seed (both classes present for n >= 2)."""
    r = (np.random.default_rng(seed).random(n) < 0.5).astype(np.uint8)
    if n >= 2:
        r[0], r[1] = 1, 0
    return r


def random_set(rng, n, escapes):
    """Short patterns over a small alphabet in random case, with lines repeated in other cases (collisions within
    and across rule classes), bytes 0xC1-0xDA and letterless lines."""
    alpha = np.frombuffer(b"abAB-1\xc1\xe1", dtype=np.uint8)
    pats = []
    for _ in range(n):
        if pats and rng.random() < 0.35:
            pats.append(random_case(pats[int(rng.integers(0, len(pats)))], int(rng.integers(0, 1 << 30))))
        else:
            pats.append(bytes(alpha[rng.integers(0, len(alpha), int(rng.integers(1, 5)))]))
    blob = octal_file(pats) if escapes else b"".join(p + b"\n" for p in pats)
    return pats, blob


@pytest.mark.parametrize("escapes", [False, True])
def test_reference_equals_brute_force(escapes):
    rng = np.random.default_rng(7 + escapes)
    alpha = np.frombuffer(b"abAB-1\xc1\xe1", dtype=np.uint8)
    for k in range(25):
        pats, blob = random_set(rng, int(rng.integers(2, 30)), escapes)
        assert patterns_of(blob, escapes) == pats
        rules = alternating(len(pats), k)
        text = alpha[rng.integers(0, len(alpha), 3000)]
        pos, ids = CaseRulesRef(blob, rules, escapes=escapes).scan(text)
        bp, bi = brute_force(pats, rules, text)
        assert np.array_equal(pos, bp) and np.array_equal(ids, bi), k


def test_get_group_reports_every_live_line_in_id_order():
    """Exact GET (1) and caseless get (2) both report on GET; only line 2 on get."""
    blob = b"GET\nget\n"
    pos, ids = CaseRulesRef(blob, [0, 1]).scan(np.frombuffer(b"GET get", dtype=np.uint8))
    assert pos.tolist() == [0, 0, 4] and ids.tolist() == [1, 2, 2]


@pytest.mark.parametrize("escapes", [False, True])
@pytest.mark.parametrize("n_parts", [1, 3])
def test_uniform_rules_are_the_uniform_sets(tmp_path, escapes, n_parts):
    from pfac_synth import synth_patterns
    pats = random_case(synth_patterns(4, 400, 17, 3, 20) + b"GET /\nget /\n", 3)
    n = len(patterns_of(pats, escapes))
    for rule, caseless in ((1, True), (0, False)):
        a = pf.Tables.from_bytes(pats, n_parts, 256, escapes=escapes, caseless=[rule] * n)
        b = pf.Tables.from_bytes(pats, n_parts, 256, escapes=escapes, caseless=caseless)
        same_tables(a, b)
        assert lib.pfac_tables_flags(a._h) == lib.pfac_tables_flags(b._h)
        assert a.source_hash() == b.source_hash() and a.caseless == caseless
        assert a.case_rules.tolist() == [rule] * n
        a.save(tmp_path / "a.bin")
        b.save(tmp_path / "b.bin")
        assert (tmp_path / "a.bin").read_bytes() == (tmp_path / "b.bin").read_bytes()


@pytest.mark.parametrize("n_parts", [1, 4])
def test_mixed_tables_are_the_caseless_tables(n_parts):
    from pfac_synth import synth_patterns
    pats = random_case(synth_patterns(6, 700, 19, 3, 30) + b"GET /\nget /\nGet /\n\xc1\xdaZ\n", 5)
    n = pats.count(b"\n")
    t = pf.Tables.from_bytes(pats, n_parts, 256, caseless=alternating(n, 1))
    assert lib.pfac_tables_flags(t._h) == pf.PFAC_PATTERNS_CASE_RULES and not t.caseless
    same_tables(t, pf.Tables.from_bytes(pats, n_parts, 256, caseless=True))
    assert t.case_rules.tolist() == alternating(n, 1).tolist()


def test_pattern_lengths_of_members_and_shadowed_lines():
    #        1      2      3      4      5      6      7     8
    blob = b"GET\nget\nGeT\nGET\nPOST\npost\n123\n123\n"
    rules = [0, 1, 0, 0, 1, 1, 0, 0]
    t = pf.Tables.from_bytes(blob, 1, 256, caseless=rules)
    # shadowed: 1 (exact GET again at 4), 5 (caseless post at 6), 7 (exact 123 at 8)
    assert t.pattern_lengths().tolist() == [0, 0, 3, 3, 3, 0, 4, 0, 3]
    # the caseless build reports the owners only
    assert pf.Tables.from_bytes(blob, 1, 256, caseless=True).pattern_lengths().tolist() == [0, 0, 0, 0, 3, 0, 4, 0, 3]


def test_case_rules_of_every_kind_of_set(tmp_path):
    blob = b"ab\nAB\ncd\n"
    assert pf.Tables.from_bytes(blob, 1, 256).case_rules.tolist() == [0, 0, 0]
    assert pf.Tables.from_bytes(blob, 1, 256, caseless=True).case_rules.tolist() == [1, 1, 1]
    t = pf.Tables.from_bytes(blob, 1, 256, caseless=[True, False, True])
    assert t.case_rules.tolist() == [1, 0, 1]
    t.save(tmp_path / "m.bin")
    assert pf.Tables.load(tmp_path / "m.bin").case_rules.tolist() == [1, 0, 1]
    p = t.part(0)
    arr = pf.Tables.from_arrays(p.s0, p.r, p.HT, p.val, 256, p.state_num, p.n_final, p.idmap, t.max_pat_len)
    assert arr.case_rules.tolist() == [0] * arr.n_patterns
    out = np.zeros(2, dtype=np.uint8)
    assert lib.pfac_tables_case_rules(t._h, out.ctypes.data, 2) == PFAC_ERR_ARG
    assert b"2 for 3 patterns" in lib.pfac_last_error()


def _build_rules(blob, flags, rules, n):
    h = C.c_void_p()
    ptr = rules.ctypes.data if rules is not None else None
    rc = lib.pfac_tables_build_mem_rules(blob, len(blob), 1, 256, flags, ptr, n, C.byref(h))
    if rc == 0:
        lib.pfac_tables_destroy(h)
    return rc, lib.pfac_last_error().decode()


def test_every_refusal_names_its_numbers(tmp_path):
    blob = b"ab\nAB\ncd\n"
    r = np.array([1, 0, 1], dtype=np.uint8)
    rc, msg = _build_rules(blob, pf.PFAC_PATTERNS_CASELESS, r, 3)
    assert rc == PFAC_ERR_ARG and "0x2" in msg and "3 patterns" in msg
    rc, msg = _build_rules(blob, pf.PFAC_PATTERNS_CASELESS | pf.PFAC_PATTERNS_ESCAPES, r, 3)
    assert rc == PFAC_ERR_ARG and "0x3" in msg
    rc, msg = _build_rules(blob, pf.PFAC_PATTERNS_CASE_RULES, r, 3)
    assert rc == PFAC_ERR_ARG and "0x4" in msg
    rc, msg = _build_rules(blob, 0, None, 3)
    assert rc == PFAC_ERR_ARG and "NULL" in msg and "3" in msg
    rc, msg = _build_rules(blob, 0, np.array([1, 2, 0], dtype=np.uint8), 3)
    assert rc == PFAC_ERR_ARG and "caseless[1] = 2" in msg
    for n in (2, 4):
        rc, msg = _build_rules(blob, 0, np.array([1, 0, 1, 0], dtype=np.uint8), n)
        assert rc == PFAC_ERR_ARG and f"{n} rules for 3 patterns" in msg
    # with escapes: one rule per decoded pattern ("a\\nb" is one pattern)
    rc, msg = _build_rules(b"a\\nb\nc\n", pf.PFAC_PATTERNS_ESCAPES, np.array([1, 0, 1], dtype=np.uint8), 3)
    assert rc == PFAC_ERR_ARG and "3 rules for 2 patterns" in msg
    assert _build_rules(b"a\\nb\nc\n", pf.PFAC_PATTERNS_ESCAPES, np.array([1, 0], dtype=np.uint8), 2)[0] == 0
    # the file and hash calls refuse the same
    f = tmp_path / "p.txt"
    f.write_bytes(blob)
    h = C.c_void_p()
    assert lib.pfac_tables_build_file_rules(str(f).encode(), 1, 256, 0, None, 3, C.byref(h)) == PFAC_ERR_ARG
    with pytest.raises(pf.PfacError, match="2 rules for 3 patterns"):
        pf.pattern_file_hash(f, caseless=[True, False])
    with pytest.raises(pf.PfacError, match="4 rules for 3 patterns"):
        pf.Tables.from_file(f, caseless=[True, False, True, False])


def test_hash_follows_every_rule(tmp_path):
    f = tmp_path / "p.txt"
    blob = b"GET\nHost\nabc\nxyz\n"
    f.write_bytes(blob)
    base = [1, 0, 1, 0]
    h0 = pf.pattern_file_hash(f, caseless=base)
    assert pf.Tables.from_file(f, caseless=base).source_hash() == h0
    assert pf.Tables.from_bytes(blob, caseless=base).source_hash() == h0
    seen = {h0, pf.pattern_file_hash(f), pf.pattern_file_hash(f, caseless=True)}
    for i in range(4):
        r = list(base)
        r[i] ^= 1
        h = pf.pattern_file_hash(f, caseless=r)
        assert h not in seen and pf.Tables.from_file(f, caseless=r).source_hash() == h
        seen.add(h)
    assert pf.pattern_file_hash(f, caseless=[1] * 4) == pf.pattern_file_hash(f, caseless=True)
    assert pf.pattern_file_hash(f, caseless=[0] * 4) == pf.pattern_file_hash(f)
    assert pf.pattern_file_hash(f, escapes=True, caseless=base) != h0


def test_cache_file_of_a_mixed_set(tmp_path):
    pats = random_case(b"GET /\nget /\nHost: \nHOST: \nabc\n123\n", 2)
    rules = [1, 0, 0, 1, 0, 0]
    t = pf.Tables.from_bytes(pats, 2, 256, caseless=rules)
    f = tmp_path / "m.bin"
    t.save(f)
    raw = f.read_bytes()
    assert raw[:8] == b"PFACTBL3" and struct.unpack_from("<I", raw, 32)[0] == pf.PFAC_PATTERNS_CASE_RULES
    assert raw[36:42] == bytes(rules)
    u = pf.Tables.load(f)
    same_tables(u, t)
    assert u.case_rules.tolist() == rules and u.source_hash() == t.source_hash()
    assert lib.pfac_tables_flags(u._h) == pf.PFAC_PATTERNS_CASE_RULES
    for g in range(2):
        assert np.array_equal(u.pattern_lengths(g), t.pattern_lengths(g))
    u.save(tmp_path / "again.bin")
    assert (tmp_path / "again.bin").read_bytes() == raw
    for k in (33, 37, len(raw) // 2, len(raw) - 20, len(raw) - 1):   # flags, rules, arrays, verify tables, checksum
        bad = bytearray(raw)
        bad[k] ^= 0x21
        g = tmp_path / f"bad{k}.bin"
        g.write_bytes(bytes(bad))
        with pytest.raises(pf.PfacError):
            pf.Tables.load(g)
    for cut in (40, len(raw) - 30, len(raw) - 1):
        g = tmp_path / f"short{cut}.bin"
        g.write_bytes(raw[:cut])
        with pytest.raises(pf.PfacError):
            pf.Tables.load(g)


def test_filter_profile_of_a_mixed_set_counts_the_folded_text():
    from pfac_synth import synth_patterns, synth_text
    pats = synth_patterns(2, 800, 31, 4, 24)
    text = random_case(synth_text(2, 33, 100000, patterns=pats), 4)
    n = pats.count(b"\n")
    mixed = pf.Tables.from_bytes(random_case(pats, 5), 1, 256, caseless=alternating(n, 2))
    assert mixed.filter_profile(text) == pf.Tables.from_bytes(fold(pats), 1, 256).filter_profile(fold(text))


# ---------------------------------------------------------------- the CLI's GPHF_NOCASE_LINES (refusals need no GPU)

def _cli(tmp_path, pats, lines, **env):
    pat, inp, nc = tmp_path / "pats", tmp_path / "in", tmp_path / "nocase"
    pat.write_bytes(pats)
    inp.write_bytes(b"GET get xyz\n")
    nc.write_bytes(lines)
    return subprocess.run([GPHF, str(pat), "1", "256", str(inp)], cwd=tmp_path, capture_output=True, text=True,
                          env=dict(os.environ, GPHF_NOCASE_LINES=str(nc), **env))


@pytest.mark.parametrize("lines,why", [
    (b"1\nx\n", "line 2 of"), (b"1\n\n2\n", "line 2 of"), (b"1 \n", "line 1 of"), (b"-1\n", "line 1 of"),
    (b"0\n", "pattern 0 (line 1"), (b"4\n", "pattern 4 (line 1"), (b"2\n99999999999999999999\n", "(line 2"),
])
def test_cli_refuses_bad_nocase_lines(tmp_path, lines, why):
    r = _cli(tmp_path, b"GET\nget\nxyz\n", lines)
    assert r.returncode == 1 and why in r.stderr, r.stderr


def test_cli_counts_patterns_like_the_reader(tmp_path):
    """The range check uses the reader's pattern count: with escapes, a newline that \\x skips as white space ends
    no pattern."""
    r = _cli(tmp_path, b"a\\x\nb\nc\\\nd\n", b"4\n", GPHF_ESCAPES="1")
    assert r.returncode == 1 and "the file has 3 patterns" in r.stderr, r.stderr
    r = _cli(tmp_path, b"a\\x\nb\nc\\\nd\n", b"4\n")
    assert r.returncode == 1 and "the file has 4 patterns" not in r.stderr   # (in range: it gets past the parse)


def test_cli_refuses_nocase_lines_with_caseless(tmp_path):
    r = _cli(tmp_path, b"GET\nget\n", b"1\n", GPHF_CASELESS="1")
    assert r.returncode == 1 and "exclude each other" in r.stderr
