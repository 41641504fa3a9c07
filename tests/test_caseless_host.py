"""Caseless pattern sets (PFAC_PATTERNS_CASELESS) on the host: the fold rule, the tables, the cache formats, the
source hash and the filter profile -- and the helpers the GPU tests (tests/test_caseless_gpu.py) share.

The definition every test checks: scan(tables of P built caseless, T) == scan(tables of fold(P), fold(T)), where fold
maps 'A'-'Z' (0x41-0x5A) to 'a'-'z' and leaves every other byte, 0xC1-0xDA included, as it is."""
import copy
import struct

import numpy as np
import pytest

import phfpfac_b200 as pf
from _caseless_ref import FOLD, FOLD_NP, caseless_oracle, decode_escapes, fold, octal_file
from _oracle import Oracle
from test_detector_paths_host import CASES, get_case, lines_of


def random_case(data, seed):
    """Every ASCII letter of data in upper or lower case at random; no other byte changes (fold(random_case(x)) ==
    fold(x)).  bytes -> bytes, uint8 array -> a new array."""
    arr = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    rng = np.random.default_rng(seed)
    low = FOLD_NP[arr]
    letter = (low >= 0x61) & (low <= 0x7A)
    up = letter & (rng.random(len(arr)) < 0.5)
    out = np.where(up, low - 0x20, low).astype(np.uint8)
    out = np.where(letter, out, arr).astype(np.uint8)
    return out if isinstance(data, np.ndarray) else out.tobytes()


def same_tables(a, b):
    assert a.n_parts == b.n_parts and a.n_patterns == b.n_patterns and a.max_pat_len == b.max_pat_len
    for g in range(a.n_parts):
        pa, pb = a.part(g), b.part(g)
        for k in ("state_num", "n_final", "max_len", "ht_size", "n_r", "n_keys", "max_key", "max_offset", "min_len"):
            assert getattr(pa, k) == getattr(pb, k), (g, k)
        for k in ("s0", "r", "HT", "val", "idmap"):
            assert np.array_equal(getattr(pa, k), getattr(pb, k)), (g, k)


# ---------------------------------------------------------------- detector-path cases, caseless

def _derived(tables):
    """What decides a set's detector kernel on the host: derive_check of partition 0."""
    d = tables.derive_check(0)
    return {k: d[k] for k in ("has_short", "has_t3", "prefixes4")}, d["tm2_keys"] > 0


_CASELESS_CASES = {}


def caseless_case(name):
    """The detector-path case `name` (tests/test_detector_paths_host.py) as a caseless set: its pattern file in
    random case, its tables built with caseless=True.  Its effective patterns (case.lines, the reference's set) are
    the folded lines -- or, where folding would merge lines or move the set onto another detector kernel (derive
    check), its lines with every capital replaced by the byte 0x80 above it, which does not fold, so the same path
    runs.  Texts are built from case.lines and scanned in random case; the reference scans their fold."""
    if name in _CASELESS_CASES:
        return _CASELESS_CASES[name]
    base = get_case(name)
    assert not base.spec.get("dag"), "sets wrapped from arrays are case-sensitive"
    lines = [fold(p) for p in base.lines]
    moved = len(set(lines)) != len(lines)
    if not moved:
        moved = _derived(pf.Tables.from_bytes(b"".join(p + b"\n" for p in lines), 1, 256)) != _derived(base.tables)
    if moved:
        lines = [bytes(c + 0x80 if 0x41 <= c <= 0x5A else c for c in p) for p in base.lines]
        assert len(set(lines)) == len(lines)
    case = copy.copy(base)
    case.moved = moved
    case.lines = lines
    case.blob = b"".join(p + b"\n" for p in lines)
    case.file = random_case(case.blob, 1000 + len(name))
    case.tables = pf.Tables.from_bytes(case.file, 1, 256, caseless=True)
    case.rp = fold(base.rp) if not moved else bytes(c + 0x80 if 0x41 <= c <= 0x5A else c for c in base.rp)
    case._oracle = None
    _CASELESS_CASES[name] = case
    return case


CASELESS_CASES = [k for k, v in CASES.items() if not v.get("dag")]


# ---------------------------------------------------------------- tests

def test_fold_rule_over_every_byte_value():
    """The Python fold, the builder's and the oracle's agree on all 256 byte values: only 0x41-0x5A change."""
    for b in range(256):
        want = b + 0x20 if 0x41 <= b <= 0x5A else b
        assert FOLD[b] == want
    # every non-newline byte value as a one-byte pattern: the caseless set is the set of the folded bytes
    blob = b"".join(bytes([b]) + b"\n" for b in range(256) if b != 10)
    t = pf.Tables.from_bytes(blob, 1, 256, caseless=True)
    same_tables(t, pf.Tables.from_bytes(fold(blob), 1, 256))
    o = caseless_oracle(blob, 1, 256)
    text = np.arange(256, dtype=np.uint8)
    pos, ids = o.scan(fold(text))
    want_pos, want_ids = Oracle(fold(blob), 1, 256).scan(fold(text))
    assert np.array_equal(pos, want_pos) and np.array_equal(ids, want_ids)
    # 0xC1-0xDA match only themselves: no fold of the high half
    hi = {int(p): int(i) for p, i in zip(pos, ids) if p >= 0xC1 and p <= 0xDA}
    assert all(blob.split(b"\n")[hi[p] - 1] == bytes([p]) for p in hi)


@pytest.mark.parametrize("width", [1, 16, 64, 256, 4096])
@pytest.mark.parametrize("n_parts", [1, 3, 4])
def test_caseless_tables_are_the_tables_of_the_folded_file(width, n_parts):
    from pfac_synth import synth_patterns
    pats = synth_patterns(5, 600, 21, 3, 30) + b"GET /\nget /\nHost: \nHOST: \n\xc1\xdaZ\n"
    file = random_case(pats, width + n_parts)
    t = pf.Tables.from_bytes(file, n_parts, width, caseless=True)
    assert t.caseless
    same_tables(t, pf.Tables.from_bytes(fold(file), n_parts, width))
    if width < 64:   # (the reference's fixed-size hash table of the oracle overflows at narrow widths)
        return
    # and the same as the oracle's caseless build
    o = caseless_oracle(file, n_parts, width)
    assert o.n_patterns == t.n_patterns and o.max_pat_len == t.max_pat_len
    for g in range(n_parts):
        assert o.part(g).same_as(t.part(g)), g


def test_escapes_with_caseless_follow_the_oracle():
    """The fold comes after the escape reader: \\x41 is 'A', then 'a'; \\x61 stays 'a'; \\\\ stays a backslash.
    Folding the raw file instead would leave \\x41 as 'A'."""
    file = b"\\x41BC\n\\x61bc\nX\\\\Y\n\\101\\x5a\n\\xc1q\nz\\tW\n"
    t = pf.Tables.from_bytes(file, 1, 256, escapes=True, caseless=True)
    o = caseless_oracle(file, 1, 256, escapes=True)
    text = random_case(np.frombuffer(b"..aBc..ABC..x\\y..az..\xc1Q..\xe1q..Z\tw..", dtype=np.uint8), 3)
    pos, ids = o.scan(fold(text))
    # ids: 'abc' (lines 1 and 2 merge, line 2 wins), 'x\\y', 'az', '\xc1q', 'z\tw'
    got = sorted(zip(pos.tolist(), ids.tolist()))
    assert [i for _, i in got] == [2, 2, 3, 4, 5, 6], got
    # the tables equal the oracle's (its canonical arrays)
    from _oracle import scan_tables_cpu
    p = t.part(0)
    cpos, cids = scan_tables_cpu(p, p.idmap, t.max_pat_len, fold(text))
    assert np.array_equal(cpos, pos) and np.array_equal(cids, ids)
    # folding the raw file is NOT the same set: \x41 would still read as 'A'
    raw = pf.Tables.from_bytes(fold(file), 1, 256, escapes=True)
    q = raw.part(0)
    rpos, rids = scan_tables_cpu(q, q.idmap, raw.max_pat_len, fold(text))
    assert sorted(zip(rpos.tolist(), rids.tolist())) != got


def test_duplicates_after_folding_report_the_last_line():
    t = pf.Tables.from_bytes(b"GET\nget\nGet\nPOST\n", 1, 256, caseless=True)
    lens = t.pattern_lengths()
    assert lens.tolist() == [0, 0, 0, 3, 4]
    from _oracle import scan_tables_cpu
    p = t.part(0)
    pos, ids = scan_tables_cpu(p, p.idmap, t.max_pat_len, np.frombuffer(fold(b"xGeT get POST"), dtype=np.uint8))
    assert pos.tolist() == [1, 5, 9] and ids.tolist() == [3, 3, 4]
    o = caseless_oracle(b"GET\nget\nGet\nPOST\n", 1, 256)
    opos, oids = o.scan(np.frombuffer(fold(b"xGeT get POST"), dtype=np.uint8))
    assert np.array_equal(opos, pos) and np.array_equal(oids, ids)


def test_source_hash_differs_per_flag(tmp_path):
    f = tmp_path / "p.txt"
    f.write_bytes(b"Abc\n\\x41d\n")
    hashes = {(e, c): pf.pattern_file_hash(f, escapes=e, caseless=c) for e in (False, True) for c in (False, True)}
    assert len(set(hashes.values())) == 4
    for (e, c), h in hashes.items():
        assert pf.Tables.from_file(f, 1, 256, escapes=e, caseless=c).source_hash() == h


def test_cache_formats(tmp_path):
    """Case-sensitive sets write PFACTBL2 (unchanged); caseless sets PFACTBL3 with the flag after the source hash,
    under the checksum; both load, PFACTBL2 as case-sensitive; a damaged PFACTBL3 is refused."""
    pats = b"GET /\nHost: \nUser-Agent\n"
    cs = pf.Tables.from_bytes(pats, 2, 256)
    ci = pf.Tables.from_bytes(pats, 2, 256, caseless=True)
    f2, f3 = tmp_path / "cs.bin", tmp_path / "ci.bin"
    cs.save(f2)
    ci.save(f3)
    b2, b3 = f2.read_bytes(), f3.read_bytes()
    assert b2[:8] == b"PFACTBL2" and b3[:8] == b"PFACTBL3"
    # PFACTBL2: magic, 4 x i32, u64 hash, then the partitions; PFACTBL3 adds u32 flags after the hash
    assert struct.unpack_from("<I", b3, 32)[0] == pf.PFAC_PATTERNS_CASELESS
    assert len(b3) == len(b2) + 4
    l2, l3 = pf.Tables.load(f2), pf.Tables.load(f3)
    assert not l2.caseless and l3.caseless
    assert l3.source_hash() == ci.source_hash() and l2.source_hash() == cs.source_hash()
    same_tables(l3, ci)
    same_tables(l2, cs)
    # the case-sensitive file is byte for byte what the cache format has always been: the same bytes as a
    # PFACTBL2 cache of the folded set except for the hash... and a caseless set of a file without capitals has
    # the same arrays as the case-sensitive one, so its PFACTBL3 file is the PFACTBL2 file plus the flag word
    lo = pats.lower()
    a, b = tmp_path / "lo2.bin", tmp_path / "lo3.bin"
    pf.Tables.from_bytes(lo, 2, 256).save(a)
    pf.Tables.from_bytes(lo, 2, 256, caseless=True).save(b)
    x, y = a.read_bytes(), b.read_bytes()
    assert x[8:24] == y[8:24] and x[32:-8] == y[36:-8]
    for k in (8, 33, len(b3) // 2, len(b3) - 1):   # a flipped byte: header, flags, arrays, checksum
        bad = bytearray(b3)
        bad[k] ^= 0x40
        g = tmp_path / f"bad{k}.bin"
        g.write_bytes(bytes(bad))
        with pytest.raises(pf.PfacError):
            pf.Tables.load(g)
    g = tmp_path / "short.bin"
    g.write_bytes(b3[:-3])
    with pytest.raises(pf.PfacError):
        pf.Tables.load(g)


def test_filter_profile_counts_the_folded_text():
    from pfac_synth import synth_patterns, synth_text
    pats = synth_patterns(2, 800, 31, 4, 24) + b"GET /index\nHost: www\n"
    text = random_case(synth_text(2, 33, 200000, patterns=pats), 4)
    ci = pf.Tables.from_bytes(random_case(pats, 5), 1, 256, caseless=True)
    cs = pf.Tables.from_bytes(fold(pats), 1, 256)
    assert ci.filter_profile(text) == cs.filter_profile(fold(text))


def test_caseless_property():
    assert pf.Tables.from_bytes(b"ab\n", 1, 256, caseless=True).caseless
    assert not pf.Tables.from_bytes(b"ab\n", 1, 256).caseless
    assert not pf.Tables.from_bytes(b"ab\n", 1, 256, escapes=True).caseless
    t = pf.Tables.from_bytes(b"ab\n", 1, 256)
    p = t.part(0)
    assert not pf.Tables.from_arrays(p.s0, p.r, p.HT, p.val, 256, p.state_num, p.n_final, p.idmap, t.max_pat_len).caseless


@pytest.mark.parametrize("name", CASELESS_CASES)
def test_caseless_detector_cases_keep_their_kernel(name):
    """Each detector-path case, made caseless, keeps the host-side signature of its kernel, and its caseless
    tables are the tables of its effective lines."""
    case = caseless_case(name)
    base = get_case(name)
    assert _derived(case.tables) == _derived(base.tables), (name, case.moved)
    same_tables(case.tables, pf.Tables.from_bytes(case.blob, 1, 256))
    assert fold(case.blob) == case.blob
    assert lines_of(case.blob) == case.lines and fold(case.file) == case.blob


def test_escape_decoder_of_the_reference_reads_like_the_oracle():
    """The caseless reference decodes escaped files itself: its decoder and octal re-encoding give the oracle's own
    escape-reader tables, on hand-made escapes and on random escape soup."""
    rng = np.random.default_rng(11)
    files = [b"\\x41BC\n\\x61bc\nX\\\\Y\n\\101\\x5a\n\\xc1q\nz\\tW\n\\q\\x 4Fk\n\\777\\0a\n\\\"\\'\\v\\f\\r\\n\\a\\b\n"]
    alphabet = np.frombuffer(b"\\x0123456789abcdefABCDEFntvr'\" qZ\t\xc1\xff", dtype=np.uint8)
    for _ in range(30):
        lines = [bytes(alphabet[rng.integers(0, len(alphabet), int(rng.integers(1, 12)))]) for _ in range(20)]
        files.append(b"".join(ln + b"x\n" for ln in lines))
    for f in files:
        a, b = Oracle(f, 1, 256, escapes=True), Oracle(octal_file(decode_escapes(f)), 1, 256, escapes=True)
        assert a.n_patterns == b.n_patterns and a.part(0).same_as(b.part(0)), f
