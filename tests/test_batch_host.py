"""Pattern lengths per id (the table the batch scan's split pass reads): host-side, no GPU."""
import ctypes as C

import numpy as np
import pytest

import phfpfac_b200 as pf
from phfpfac_b200._lib import PFAC_ERR_ARG, PFAC_ERR_OUTPUT_FULL, lib


def expected_lengths(pats, t, g):
    """Per id of partition g: the line's length if it is the last copy of its line within the partition (the
    earlier copies of a duplicated line are overwritten in the trie, create_table_reorder.c:362-366), else 0."""
    lines = pats.split(b"\n")[:-1]
    ids = [int(i) for i in t.part(g).idmap]
    last = {}
    for i in ids:
        last[lines[i - 1]] = max(last.get(lines[i - 1], 0), i)
    want = np.zeros(max(ids) + 1, dtype=np.int32)
    for text, i in last.items():
        want[i] = len(text)
    return want, ids


def check_lengths(pats, n_parts=1, width=256):
    t = pf.Tables.from_bytes(pats, n_parts=n_parts, width=width)
    for g in range(t.n_parts):
        got = t.pattern_lengths(g)
        want, ids = expected_lengths(pats, t, g)
        assert np.array_equal(got, want), g
        assert (got[ids] > 0).sum() == len(set(pats.split(b"\n")[i - 1] for i in ids))
    return t


@pytest.mark.parametrize("name", ["experimentpattern", "xad"])
def test_pattern_lengths_of_fixtures(fixtures, name):
    check_lengths(fixtures[name])


def test_pattern_lengths_random_set_with_duplicates():
    rng = np.random.default_rng(7)
    base = [bytes(rng.integers(97, 101, int(rng.integers(1, 12))).astype(np.uint8)) for _ in range(400)]
    lines = base + [base[int(i)] for i in rng.integers(0, len(base), 200)]
    rng.shuffle(lines)
    pats = b"".join(p + b"\n" for p in lines)
    t = check_lengths(pats)
    assert len(set(lines)) < len(lines)
    got = t.pattern_lengths()
    assert (got == 0).sum() >= len(lines) - len(set(lines))   # every earlier copy of a line reports nothing


def test_pattern_lengths_multi_partition(fixtures):
    """Ids are global line numbers: a partition's ids run far beyond its own n_final."""
    pats = fixtures["xad"]
    t = check_lengths(pats, n_parts=8, width=64)
    p = t.part(7)
    assert len(t.pattern_lengths(7)) > p.n_final


def test_pattern_lengths_refuses_a_dag():
    t = pf.Tables.from_bytes(b"abc\nacd\nbx\nzz\n")
    p = t.part(0)
    s0 = p.s0.copy()
    s0[ord("b")] = s0[ord("a")]                  # two root edges into one state: no single depth
    dag = pf.Tables.from_arrays(s0, p.r, p.HT, p.val, 256, p.state_num, p.n_final, p.idmap, p.max_len)
    with pytest.raises(pf.PfacError) as e:
        dag.pattern_lengths()
    assert e.value.code == PFAC_ERR_ARG
    n = C.c_int32(0)
    assert lib.pfac_tables_pattern_lengths(dag._h, 0, None, 0, C.byref(n)) == PFAC_ERR_ARG


def test_pattern_lengths_query_and_capacity():
    pats = b"abc\nab\nabc\nxyz\nq\n"
    t = pf.Tables.from_bytes(pats)
    n = C.c_int32(0)
    assert lib.pfac_tables_pattern_lengths(t._h, 0, None, 0, C.byref(n)) == 0
    assert n.value == 6                          # max id (line 5) + 1
    small = np.full(5, -7, dtype=np.int32)
    assert lib.pfac_tables_pattern_lengths(t._h, 0, small.ctypes.data, 5, C.byref(n)) == PFAC_ERR_OUTPUT_FULL
    big = np.full(9, -7, dtype=np.int32)
    assert lib.pfac_tables_pattern_lengths(t._h, 0, big.ctypes.data, 9, C.byref(n)) == 0
    assert n.value == 6
    assert big.tolist() == [0, 0, 2, 3, 3, 1, 0, 0, 0]   # line 1 "abc" is overwritten by its copy on line 3
    assert lib.pfac_tables_pattern_lengths(t._h, 1, None, 0, C.byref(n)) == PFAC_ERR_ARG   # no partition 1
