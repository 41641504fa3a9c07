"""The product's table builder (phfpfac_b200/csrc/pfac_tables.cc) is bit-compatible with
create_PFAC_table_reorder + FFDM: compared with the reference-generated goldens, with the oracle
on random sets, and (where oracle/_ref exists) with the reference builder itself."""
import os

import numpy as np
import pytest

import phfpfac_b200 as pf
import pfac_synth as synth
from _oracle import Oracle, RefBuild, ref_available
from _ref_sets import product_builder_sets, random_patterns
from conftest import digest, parse_key


def same(a, b):
    return (a.state_num == b.state_num and a.n_final == b.n_final and a.max_len == b.max_len
            and a.ht_size == b.ht_size and np.array_equal(a.s0, b.s0) and np.array_equal(a.r, b.r)
            and np.array_equal(a.HT, b.HT) and np.array_equal(a.val, b.val) and np.array_equal(a.idmap, b.idmap))


def test_tables_match_reference_goldens(fixtures, golden):
    for key, g in golden["ref_tables"].items():
        name, parts, width = parse_key(key)
        t = pf.Tables.from_bytes(fixtures[name], n_parts=parts, width=width)
        assert t.n_parts == parts and t.max_pat_len == g["max_pat_len"], key
        for i, want in enumerate(g["parts"]):
            assert digest(t.part(i)) == want, (key, i)


def test_kat_counts(fixtures, golden):
    for name, k in golden["kat_counts"].items():
        p = pf.Tables.from_bytes(fixtures[name], n_parts=1, width=k["width"]).part(0)
        assert (p.state_num, p.n_final, p.n_keys, p.max_key) == (k["state_num"], k["n_final"], k["n_keys"], k["max_key"])


@pytest.mark.parametrize("seed", range(8))
def test_tables_equal_oracle_random(seed):
    rng = np.random.default_rng(100 + seed)
    n = int(rng.integers(1, 1500))
    blob = random_patterns(rng, n, int(rng.integers(1, 200)) if seed % 2 else int(rng.integers(2, 6)),
                           int(rng.integers(1, 40)), base=11 if seed % 2 else 97)
    width = int(2 ** rng.integers(5, 13))
    parts = int(rng.integers(1, 9))
    if parts > n:
        parts = 1
    o = Oracle(blob, n_parts=parts, width=width)
    t = pf.Tables.from_bytes(blob, n_parts=parts, width=width)
    assert t.n_patterns == o.n_patterns and t.max_pat_len == o.max_pat_len
    for g in range(parts):
        a, b = t.part(g), o.part(g)
        assert same(a, b), (seed, g)
        assert a.n_keys == b.extra["n_keys"] and a.max_key == b.extra["max_key"] and a.max_offset == b.extra["max_offset"]


def test_duplicate_and_prefix_patterns():
    """Duplicates: the last in sort order owns the final state (create_table_reorder.c:366);
    prefixes: the shorter pattern's final state becomes an interior node (:116)."""
    blob = b"abc\nab\nabc\nabcd\na\nabc\nb\n"
    for parts in (1, 2):
        o = Oracle(blob, n_parts=parts, width=64)
        t = pf.Tables.from_bytes(blob, n_parts=parts, width=64)
        for g in range(parts):
            assert same(t.part(g), o.part(g))


def test_lookup_equals_transition_rule(fixtures):
    """pfac_tables_lookup == master_kernel.cu:52-64 over the canonical arrays == the trie edge."""
    o = Oracle(fixtures["xad"], n_parts=1, width=256)
    t = pf.Tables.from_bytes(fixtures["xad"], n_parts=1, width=256)
    p = t.part(0)
    rng = np.random.default_rng(3)
    for s in rng.integers(0, p.state_num, 64):
        row = o.pfac_row(0, int(s))
        for b in rng.integers(0, 256, 32):
            assert t.lookup(int(s), int(b)) == row[int(b)]
        for b in np.nonzero(row >= 0)[0]:
            assert t.lookup(int(s), int(b)) == row[int(b)]
    assert t.lookup(p.state_num + 5, 0) == -1 and t.lookup(-1, 3) == -1


def test_from_arrays_roundtrip(fixtures):
    t = pf.Tables.from_bytes(fixtures["xad"], n_parts=1, width=128)
    p = t.part(0)
    t2 = pf.Tables.from_arrays(p.s0, p.r, p.HT, p.val, 128, p.state_num, p.n_final, p.idmap, p.max_len)
    q = t2.part(0)
    assert same(p, q) and t2.max_pat_len == t.max_pat_len and t2.n_parts == 1


def test_from_arrays_rejects_inconsistent_tables(fixtures):
    """The kernels index r[] / {HT,val} / s0 with what the arrays hold, unchecked (as the reference does):
    arrays that did not come out of the builder are checked once, at the boundary."""
    t = pf.Tables.from_bytes(fixtures["xad"], n_parts=1, width=128)
    p = t.part(0)

    def wrap(**kw):
        a = dict(s0=p.s0.copy(), r=p.r.copy(), HT=p.HT.copy(), val=p.val.copy(), width=128, state_num=p.state_num,
                 n_final=p.n_final, idmap=p.idmap.copy(), max_len=p.max_len)
        a.update(kw)
        return pf.Tables.from_arrays(a["s0"], a["r"], a["HT"], a["val"], a["width"], a["state_num"], a["n_final"],
                                     a["idmap"], a["max_len"])

    wrap()
    bad_val = p.val.copy()
    bad_val[np.argmax(bad_val >= 0)] = p.state_num + 7            # a next state that does not exist
    bad_s0 = p.s0.copy()
    bad_s0[65] = p.state_num
    bad_ht = p.HT.copy()
    bad_ht[np.argmax(bad_ht >= 0)] = len(p.r) + 3                 # a row id past r[]
    for kw in (dict(val=bad_val), dict(s0=bad_s0), dict(HT=bad_ht), dict(r=p.r[:-1].copy()), dict(max_len=-1),
               dict(state_num=p.state_num + 1)):
        with pytest.raises(pf.PfacError):
            wrap(**kw)


def test_error_behaviour(tmp_path):
    """Library errors instead of the reference's exit()/UB (create_table_reorder.c:71-77,:362; phf.c:161)."""
    cases = [(b"abc\n\nabd\n", 256, -3), (b"abc\nabd", 256, -2), (b"x" * 1023 + b"\n", 256, -2),
             (b"abc\n", 100, -4), (b"abc\n", 8192, -4), (b"abc\n", 0, -4), (b"", 256, -2)]
    for blob, width, code in cases:
        with pytest.raises(pf.PfacError) as e:
            pf.Tables.from_bytes(blob, n_parts=1, width=width)
        assert e.value.code == code, (blob[:10], width)
    with pytest.raises(pf.PfacError) as e:
        pf.Tables.from_file(str(tmp_path / "missing"), 1, 256)
    assert e.value.code == -1
    f = tmp_path / "pats"
    f.write_bytes(b"x" * 1022 + b"\nhello\n")
    t = pf.Tables.from_file(str(f), 1, 4096)
    assert t.n_patterns == 2 and t.max_pat_len == 1022


def test_large_set_beyond_reference_limits():
    """100k patterns at width 256 exceed ROW_MAX (phf.c:7): the builder has dynamic limits; the PHF
    must still be a perfect hash of the trie (every edge found, nothing else)."""
    blob = synth.synth_patterns(0, 30000, 5, 8, 32)
    t = pf.Tables.from_bytes(blob, n_parts=1, width=256)
    p = t.part(0)
    assert p.n_final == 30000 and p.n_r == p.state_num * 256 // 256 + 1
    occupied = p.HT >= 0
    assert int(occupied.sum()) == p.n_keys
    # every pattern walks to its own final state through the PHF
    lines = blob.split(b"\n")[:-1]
    order = sorted(range(len(lines)), key=lambda i: lines[i])
    for rank in (0, 1, 777, 29999):
        pat = lines[order[rank]]
        s = int(p.s0[pat[0]])
        for b in pat[1:]:
            s = t.lookup(s, b)
            assert s >= 0
        assert s == rank and p.idmap[s] == order[rank] + 1


def test_tables_equal_live_reference_builder(ref_live, tmp_path):
    """Random sets in 4 partitions and as one automaton: the reference builder's tables as stored in
    tests/golden/ref_live.json, and the live builder too where oracle/_ref was built."""
    live = ref_available()
    for trial, (blob, width) in enumerate(product_builder_sets()):
        want = ref_live["product_builder"][trial]
        assert want["width"] == width, trial
        t = pf.Tables.from_bytes(blob, n_parts=4, width=width)
        t1 = pf.Tables.from_bytes(blob, n_parts=1, width=width)
        assert [digest(t.part(g)) for g in range(4)] == want["parts"], trial
        assert digest(t1.part(0)) == want["single"], trial
        if live:
            f = tmp_path / f"p{trial}"
            f.write_bytes(blob)
            rb = RefBuild(str(f), streamnum=1, width=width)
            for g in range(4):
                assert same(t.part(g), rb.part(g)), (trial, g)
            assert same(t1.part(0), RefBuild(str(f), width=width, single=True).part(0))


@pytest.mark.parametrize("case", ["experimentpattern", "xad", "dictionary", "short", "config3", "binary"])
def test_derived_device_tables_selfcheck(fixtures, case):
    """The kernel's shared-memory accelerators (pfac_derive.cc), built and verified on the host:
    T1 exact over 2-byte prefixes, T1s/T2 supersets, hot rows == master_kernel.cu:52-64 lookups."""
    blob = {"short": b"a\nab\nabc\nabcd\nb\nbcdef\nxyzxyzxyz\n",
            "config3": synth.synth_patterns(1, 3000, 3, 4, 64),
            "binary": b"".join(bytes([i, (i * 7) % 256 or 1, 200, 201, 202]).replace(b"\n", b"\x0b") + b"\n" for i in range(256) if i != 10),
            }.get(case) or fixtures[case]
    for width in (256, 64, 4096):
        t = pf.Tables.from_bytes(blob, 1, width)
        for t2b, t3b, tm2b in ((32768, 32768, 32768), (1024, 1024, 2048), (0, 0, 0), (65536, 0, 1024), (4096, 65536, 0),
                               (0, 16384, 128)):
            st = t.derive_check(0, t2b, t3b, tm2b)
            assert st["t1_pairs"] > 0
            if t3b == 0:
                assert st["has_t3"] == 0 and st["tm_keys"] == 0
    p = pf.Tables.from_bytes(blob, 1, 256).part(0)
    t2 = pf.Tables.from_arrays(p.s0, p.r, p.HT, p.val, 256, p.state_num, p.n_final, p.idmap, p.max_len)
    assert t2.derive_check() == pf.Tables.from_bytes(blob, 1, 256).derive_check()


def test_third_window_planes_and_pattern_directory(monkeypatch):
    """Stage 1 with the third-window planes (P45 / P56 / ShX) and without (PFAC_NO_W3): both pass every pattern at
    both alignments whatever follows it (derive_check), and the third window only ever removes survivors.  The
    pattern directory of the candidate walks is checked against the walk inside derive_check as well: sets
    where it applies (trees, patterns <= 64 bytes), where it does not (a 100-byte pattern), patterns of every
    length 4..9 (the short-pattern exceptions), nested and duplicate patterns."""
    edge = b"".join(bytes([65 + (i * 7 + k) % 26 for k in range(L)]) + b"\n" for L in range(4, 10) for i in range(40))
    edge += b"GET /index\nGET /in\nGET /index.html\nGET /in\n" + b"x" * 100 + b"\n"
    sets = {"config3": synth.synth_patterns(1, 3000, 3, 4, 64), "edge": edge, "config2": synth.synth_patterns(0, 500, 1, 8, 32)}
    text = synth.synth_text(1, 4, 1 << 20, patterns=sets["config3"])
    surv = {}
    for off in (False, True):
        if off:
            monkeypatch.setenv("PFAC_NO_W3", "1")
        for name, blob in sets.items():
            t = pf.Tables.from_bytes(blob, 1, 256)
            for budget in ((32768, 32768, 32768), (1024, 1024, 2048)):
                t.derive_check(0, *budget)
            if name == "config3":
                surv[off] = t.filter_profile(text, 0, 32768, 32768, 32768)
    monkeypatch.delenv("PFAC_NO_W3")
    assert surv[False]["to_emit"] <= surv[True]["to_emit"]
    assert surv[False]["t1_pass"] < 0.9 * surv[True]["t1_pass"]      # measured: 2.6 % instead of 3.3 % of the starts


ESCAPED = (b"GET \\x2f\\x2Findex\n"          # \xhh
           b"tab\\there\n"                   # \t
           b"nul\\0byte\\101\\7z\n"          # \o, \ooo (\101 = 'A'), \7
           b"quote\\\"\\'\\\\end\n"          # \" \' \\
           b"line\\nfeed\\r\n"               # \n inside a pattern, \r
           b"not\\qescape\\\n"               # \q is not an escape: the backslash stays; trailing backslash + EOL
           b"\\a\\b\\v\\f\n"
           b"hi\\xffgh\\x7\n")               # \xff, one-digit \x7


def test_escape_front_end_matches_oracle_and_reference(tmp_path):
    """PFAC_PATTERNS_ESCAPES = read_pattern_ext / fgetc_ext (create_table_reorder.c:131-185,
    ctdef.h:37-99).  Product == oracle restatement == the reference's own reader (where built)."""
    o = Oracle(ESCAPED, n_parts=1, width=256, escapes=True)
    t = pf.Tables.from_bytes(ESCAPED, n_parts=1, width=256, escapes=True)
    assert t.n_patterns == o.n_patterns == 8
    assert same(t.part(0), o.part(0))
    # decoded bytes, checked by walking the automaton: "GET //index", "tab\there", "line\nfeed\r", ...
    p = t.part(0)
    for want in (b"GET //index", b"tab\there", b"nul\x00byteA\x07z", b"quote\"'\\end", b"line\nfeed\r",
                 b"not\\qescape\\", b"\a\b\v\f", b"hi\xffgh\x07"):
        s = int(p.s0[want[0]])
        for b in want[1:]:
            s = t.lookup(s, b)
            assert s >= 0, want
        assert s < p.n_final, want
    # without the flag the bytes are taken literally (read_pattern, the reference's live path)
    plain = pf.Tables.from_bytes(ESCAPED, n_parts=1, width=256)
    assert plain.max_pat_len > t.max_pat_len
    f = tmp_path / "esc"
    f.write_bytes(ESCAPED)
    assert same(pf.Tables.from_file(str(f), 1, 256, escapes=True).part(0), t.part(0))
    if ref_available() and os.path.isdir("/root/reference"):
        rb = RefBuild(str(f), width=256, escapes=True)
        assert same(t.part(0), rb.part(0)) and same(o.part(0), rb.part(0))
    for blob in (b"abc\\", b"\\x41", b"\n"):     # no trailing newline / empty pattern
        with pytest.raises(pf.PfacError):
            pf.Tables.from_bytes(blob, 1, 256, escapes=True)
        with pytest.raises(ValueError):
            Oracle(blob, 1, 256, escapes=True)


def test_escape_front_end_fuzz(tmp_path):
    """Random escape soup: the product's reader, the oracle's restatement and (where built) the
    reference's own read_pattern_ext agree on the tables -- or all refuse the file."""
    rng = np.random.default_rng(2024)
    atoms = [b"a", b"b", b"Z", b"0", b" ", b"\\n", b"\\t", b"\\r", b"\\0", b"\\7", b"\\12", b"\\101", b"\\377", b"\\x41",
             b"\\x4", b"\\xff", b"\\xZ", b"\\q", b"\\\\", b"\\\"", b"\\'", b"\\a", b"\\b", b"\\f", b"\\v", b"\\8", b"\\x", b"\\"]
    have_ref = ref_available() and os.path.isdir("/root/reference")
    agreed = refused = 0
    for trial in range(150):
        lines = []
        for _ in range(int(rng.integers(1, 12))):
            k = int(rng.integers(1, 7))
            lines.append(b"".join(atoms[int(i)] for i in rng.integers(0, len(atoms), k)))
        blob = b"\n".join(lines) + b"\n"
        try:
            o = Oracle(blob, 1, 256, escapes=True)
        except ValueError:
            o = None
        try:
            t = pf.Tables.from_bytes(blob, 1, 256, escapes=True)
        except pf.PfacError:
            t = None
        assert (o is None) == (t is None), (trial, blob)
        if o is None:
            refused += 1
            continue
        assert t.n_patterns == o.n_patterns and same(t.part(0), o.part(0)), (trial, blob)
        if have_ref:
            f = tmp_path / f"e{trial}"
            f.write_bytes(blob)
            assert same(t.part(0), RefBuild(str(f), width=256, escapes=True).part(0)), (trial, blob)
        agreed += 1
    assert agreed > 50


def test_table_cache_roundtrip(tmp_path, fixtures):
    """pfac_tables_save / pfac_tables_load: every canonical array of every partition comes back bit
    for bit, the derived filter tables are the same, and damaged files are refused."""
    for blob, parts, width in ((fixtures["dictionary"], 4, 64), (synth.synth_patterns(1, 3000, 3, 4, 64), 1, 256),
                               (b"a\n", 1, 4096)):
        t = pf.Tables.from_bytes(blob, parts, width)
        f = tmp_path / "cache.bin"
        t.save(f)
        u = pf.Tables.load(f)
        assert (u.n_parts, u.n_patterns, u.max_pat_len) == (t.n_parts, t.n_patterns, t.max_pat_len)
        for g in range(parts):
            a, b = t.part(g), u.part(g)
            assert same(a, b) and (a.n_keys, a.max_key, a.max_offset) == (b.n_keys, b.max_key, b.max_offset)
        assert u.derive_check() == t.derive_check()
        assert u.lookup(int(t.part(0).s0[blob[0]]), blob[1] if blob[1] != 10 else 0) == \
            t.lookup(int(t.part(0).s0[blob[0]]), blob[1] if blob[1] != 10 else 0)
    raw = bytearray(f.read_bytes())
    for damage in ("flip", "truncate", "magic"):
        bad = bytearray(raw)
        if damage == "flip":
            bad[len(bad) // 2] ^= 1
        elif damage == "truncate":
            bad = bad[:-9]
        else:
            bad[0] = ord("X")
        g = tmp_path / "bad.bin"
        g.write_bytes(bytes(bad))
        with pytest.raises(pf.PfacError) as e:
            pf.Tables.load(g)
        assert e.value.code == -1
    with pytest.raises(pf.PfacError):
        pf.Tables.load(tmp_path / "missing.bin")
    # the cache remembers what it was built from: a hash of the pattern file image and the reader flags
    pat = tmp_path / "pat"
    pat.write_bytes(fixtures["xad"])
    t = pf.Tables.from_file(str(pat), 1, 256)
    t.save(tmp_path / "c2.bin")
    u = pf.Tables.load(tmp_path / "c2.bin")
    assert u.source_hash() == t.source_hash() == pf.pattern_file_hash(str(pat)) != 0
    assert pf.pattern_file_hash(str(pat), escapes=True) != t.source_hash()
    pat.write_bytes(fixtures["xad"] + b"zzz\n")
    assert pf.pattern_file_hash(str(pat)) != u.source_hash()
    p0 = t.part(0)
    assert pf.Tables.from_arrays(p0.s0, p0.r, p0.HT, p0.val, 256, p0.state_num, p0.n_final, p0.idmap, p0.max_len).source_hash() == 0


def test_numpy_stage1_model_equals_the_cpp_model():
    """tools/host_model.py restates the detector's stage 1 in numpy to evaluate other strides / folds (DESIGN 8.1).
    Its restatement of the BUILT rule must count exactly the survivors the C++ model of the shipped tables counts."""
    import host_model as hm
    from bench import WORKLOADS
    for name in ("config3", "config2"):
        pk, cnt, pseed, lo, hi, tk, tseed, _n, _d = WORKLOADS[name]
        blob = synth.synth_patterns(pk, cnt, pseed, lo, hi)
        pats = [np.frombuffer(x, dtype=np.uint8).astype(np.uint32) for x in blob.split(b"\n")[:-1]]
        text = synth.synth_text(tk, tseed, 2 << 20, patterns=blob)
        t = pf.Tables.from_bytes(blob)
        cpp = t.filter_profile(text)
        got, n = hm.built(text, pats, True)
        # (the numpy model leaves the last 16 start positions of the text out)
        assert cpp["positions"] == len(text) == n + 16 and 0 <= cpp["t1_pass"] - got <= 16, (name, cpp["t1_pass"], got)
        # the generic (phase, window) planes are at least as selective as the built design's shared ShX plane
        ideal, _ = hm.survivors(text, pats, 2, 3)
        assert ideal <= got
