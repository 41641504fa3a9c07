"""The oracle (oracle/pfac_oracle.c) pinned against the reference: goldens generated from the
reference's own table builder (tests/golden/make_golden.py), the known-answer counts in the
reference tree, and -- where oracle/_ref was built -- the reference builder itself, live."""
import hashlib
import re

import numpy as np
import pytest

from _oracle import Oracle, RefBuild, ref_available, render_result, scan_tables_cpu
from _ref_sets import oracle_builder_sets
from conftest import digest, parse_key


def test_oracle_tables_match_reference_goldens(fixtures, golden):
    """s0Table/r/HT/val/patternIdMap of the restatement == the reference's FFDM output (golden)."""
    for key, g in golden["ref_tables"].items():
        name, parts, width = parse_key(key)
        o = Oracle(fixtures[name], n_parts=parts, width=width)
        assert o.n_parts == parts and o.max_pat_len == g["max_pat_len"], key
        for i, want in enumerate(g["parts"]):
            assert digest(o.part(i)) == want, (key, i)


def test_oracle_kat_counts_from_reference_logs(fixtures, golden):
    """experiment/xaarecord:2-6 etc. and tmp.dat:2-8: state num, final state num, keys, max key."""
    for name, k in golden["kat_counts"].items():
        o = Oracle(fixtures[name], n_parts=1, width=k["width"])
        p = o.part(0)
        assert p.state_num == k["state_num"], name
        assert p.n_final == k["n_final"], name
        assert p.extra["n_keys"] == k["n_keys"], name
        assert p.extra["max_key"] == k["max_key"], name
        if "max_len" in k:
            assert p.max_len == k["max_len"]
        if "r_size" in k:   # "r table size" = MaxKey/width + 1 (phf.c:175)
            assert p.extra["max_row"] + 1 == k["r_size"] or p.extra["max_row"] == k["r_size"], (name, p.extra, k)


@pytest.mark.parametrize("rname", ["experimentpattern_x_experimentinput", "experimentpattern_x_1M",
                                   "dictionary_x_1M", "dictionary_x_1M_single_w4096",
                                   "dictionary_x_1M_8parts_w64", "xaa_x_1M_first64k"])
def test_oracle_results_match_goldens(fixtures, golden, rname):
    g = golden["results"][rname]
    name, parts, width = parse_key(g["tables"])
    data = {"experimentpattern_x_experimentinput": fixtures["experimentinput"][:-1],
            "xaa_x_1M_first64k": fixtures["1M"][:65536]}.get(rname, fixtures["1M"][:-1])
    assert len(data) == g["input_size"]
    o = Oracle(fixtures[name], n_parts=parts, width=width)
    for dense in (False, True):
        if dense and len(data) * o.max_pat_len > 64 << 20:
            continue
        pos, ids = o.scan(data, dense=dense)
        text = render_result(pos, ids)
        assert len(pos) == g["lines"]
        assert hashlib.md5(text).hexdigest() == g["md5"]
        if "text" in g:
            assert text.decode() == g["text"]


def test_result_line_format_matches_reference_files(golden):
    """main.cc:344 "At position %4d, match pattern %d\\n" as seen in experiment/GPU_match_resultall.txt."""
    for line in golden["format_lines"]:
        m = re.fullmatch(r"At position ( *\d+), match pattern (\d+)", line)
        assert m and len(m.group(1)) >= 4
        assert render_result(np.array([int(m.group(1))]), np.array([int(m.group(2))])).decode() == line + "\n"


def test_partition_and_width_invariance(fixtures):
    """SURVEY.md 3.4: the result file does not depend on the partition count or the PHF width."""
    data = fixtures["1M"][:200000]
    base = None
    for parts, width in ((1, 256), (4, 256), (8, 64), (16, 4096), (3, 128)):
        o = Oracle(fixtures["xab"], n_parts=parts, width=width)
        pos, ids = o.scan(data)
        cur = (pos.tobytes(), ids.tobytes())
        base = base or cur
        assert cur == base, (parts, width)


def test_scan_tables_cpu_equals_partition_merge(fixtures):
    """The OpenMP walker over one partition's canonical arrays (bench.py's cpu_baseline leg)."""
    data = np.frombuffer(fixtures["1M"][:300000], dtype=np.uint8)
    o = Oracle(fixtures["dictionary"], n_parts=1, width=256)
    pos, ids = o.scan(data)
    p = o.part(0)
    for nt in (1, 3):
        pos2, ids2 = scan_tables_cpu(p, p.idmap, o.max_pat_len, data, nthreads=nt)
        assert np.array_equal(pos, pos2) and np.array_equal(ids, ids2)
    assert scan_tables_cpu(p, p.idmap, o.max_pat_len, data, nthreads=2, count_only=True) == len(pos)
    # the single-pass variant timed by bench.py (thread-local buffers, concatenated in range order),
    # also when the first capacity guess is too small
    from _oracle import scan_tables_cpu_1pass
    for nt, cap in ((1, None), (4, None), (3, 1000)):
        pos3, ids3 = scan_tables_cpu_1pass(p, p.idmap, o.max_pat_len, data, nthreads=nt, cap=cap)
        assert np.array_equal(pos, pos3) and np.array_equal(ids, ids3)


def test_oracle_error_cases():
    with pytest.raises(ValueError):
        Oracle(b"abc\n\nabd\n", 1, 256)          # empty line (create_table_reorder.c:362 UB, defined away)
    with pytest.raises(ValueError):
        Oracle(b"abc\nabd", 1, 256)              # no trailing newline (create_table_reorder.c:71-77)
    with pytest.raises(ValueError):
        Oracle(b"x" * 1023 + b"\n", 1, 256)      # "length over 1024" (create_table_reorder.c:74)
    with pytest.raises(ValueError):
        Oracle(b"abc\n", 1, 8192)                # width > COL_MAX (phf.c:161)
    Oracle(b"x" * 1022 + b"\n", 1, 4096)


def test_oracle_equals_live_reference_builder(ref_live, tmp_path):
    """Random pattern sets through the reference's own create_PFAC_table_reorder + FFDM: its tables as stored in
    tests/golden/ref_live.json, and the live builder too where oracle/_ref was built."""
    live = ref_available()
    for trial, (blob, streamnum, width) in enumerate(oracle_builder_sets()):
        want = ref_live["oracle_builder"][trial]
        assert (want["streamnum"], want["width"]) == (streamnum, width), trial
        o = Oracle(blob, n_parts=len(want["parts"]), width=width)
        assert o.max_pat_len == want["max_pat_len"], trial
        for g, d in enumerate(want["parts"]):
            assert digest(o.part(g)) == d, (trial, g, width)
        if live:
            f = tmp_path / f"p{trial}"
            f.write_bytes(blob)
            rb = RefBuild(str(f), streamnum=streamnum, width=width)
            assert rb.n_parts == o.n_parts and o.max_pat_len == rb.max_pat_len
            for g in range(rb.n_parts):
                assert o.part(g).same_as(rb.part(g)), (trial, g, width)
