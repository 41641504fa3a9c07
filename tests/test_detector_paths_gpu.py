"""Every detector kernel path against its reference, at the lane, slice, slot and tile phases, misaligned inputs, short
scan ranges and input ends where kernels go wrong.  Cases, texts and references: tests/test_detector_paths_host.py.
Each case first asserts its signature (derived mode, short patterns, level 2, launches), so a case that drifts off
its kernel fails instead of passing with less coverage."""
import numpy as np
import pytest

import phfpfac_b200 as pf
from test_detector_paths_host import (CASES, QUEUE_CASES, REF_HALO, T2_GLOBAL_BYTES, get_case, phase_text, queue_text,
                                      set_env)

pytestmark = pytest.mark.gpu

OFFSETS = (0, 1, 2, 3, 7, 8, 15)


def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def check_signature(m, case):
    spec = case.spec
    di = m.derived_info()
    assert di["mode"] == spec["mode"], (case.name, di)
    assert di["has_short"] == spec["has_short"], (case.name, di)
    assert (di["tm2_keys"] > 0) == spec["level2"], (case.name, di)
    if spec["mode"] == 2:
        assert di["t2_bits"] // 8 == T2_GLOBAL_BYTES, di
    assert case.min_len == spec["shortest"]
    # the pattern directory needs a tree and patterns of at most 64 bytes
    assert (case.max_len <= 64) == ("max_len" not in spec) and case.max_len == spec.get("max_len", case.max_len)
    if spec["kernel"].startswith("pfac_scan2_kernel<F,F"):
        assert all(len(p) >= 5 for p in case.lines)


def check_launches(m, case):
    assert m.last_info()["launches"] == case.spec["launches"], case.name


class Expect:
    """Reference records of slices of one text, from one reference scan where that is exact (patterns of at most
    513 bytes: a match is reported iff it lies inside the slice); by scanning the slice otherwise."""

    def __init__(self, case, text):
        self.case, self.text = case, text
        self.pos, self.ids = case.reference(text)
        self.end = self.pos + case.lens[self.ids - 1]

    def __call__(self, a, n_valid, n_starts=None):
        n_starts = n_valid if n_starts is None else n_starts
        if self.case.max_len > REF_HALO + 1:
            pos, ids = self.case.reference(self.text[a:a + n_valid])
        else:
            keep = (self.pos >= a) & (self.end <= a + n_valid)
            pos, ids = self.pos[keep] - a, self.ids[keep]
        keep = pos < n_starts
        return pos[keep], ids[keep]


def same(got, want, what):
    pos, ids = want
    assert len(got) == len(pos), (what, len(got), len(pos))
    assert np.array_equal(got["pos"].astype(np.int64), pos), what
    assert np.array_equal(got["id"].astype(np.int32), ids), what


@pytest.mark.parametrize("name", list(CASES))
def test_detector_path_against_reference(name, monkeypatch):
    """Plants at every phase (case.plants x phase_starts) in four layouts, near-misses, the end zone: device scans at
    seven pointer offsets, with n_starts < n_valid, at prefix lengths around the input-end bound, and a host
    scan in 16 KiB chunks -- records equal to the reference's, bit for bit."""
    torch = torch_cuda()
    case = get_case(name)
    set_env(monkeypatch, case.spec)
    m = pf.Matcher(case.tables, device=0, n_streams=2, chunk_bytes=16384)
    check_signature(m, case)
    text, info = phase_text(case)
    n = len(text)
    expect = Expect(case, text)
    assert len(expect.pos) > len(info["plants"]) // 2
    d = torch.from_numpy(text).cuda()
    for off in OFFSETS:
        got = m.scan_device(d, n_starts=n - off, n_valid=n - off, offset=off)
        check_launches(m, case)
        same(got, expect(off, n - off), (name, "offset", off))
    plant = info["plants"][len(info["plants"]) // 3]
    for ns in (n, n - 1, plant, plant + 1):
        same(m.scan_device(d, n_starts=ns, n_valid=n), expect(0, n, ns), (name, "n_starts", ns))
    # prefixes: n - max_len at -1, 0, +1 from a tile border (the longest pattern starts on it), a cut pattern
    border, L = info["border"], case.max_len
    for nn in (border + L - 1, border + L, border + L + 1, info["cut"] + info["cut_len"] - 1):
        same(m.scan_device(d, n_starts=nn, n_valid=nn), expect(0, nn), (name, "prefix", nn))
    if case.max_len > REF_HALO + 1:   # a shard that starts mid-tile keeps the global tile grid (base_pos)
        a = 5000
        got = m.scan_device(d, n_starts=n - a, n_valid=n - a, base_pos=a, offset=a)
        keep = expect.pos >= a
        same(got, (expect.pos[keep] - a, expect.ids[keep]), (name, "base_pos"))
    same(m.scan_host(text), (expect.pos, expect.ids), (name, "host"))
    m.close()


@pytest.mark.parametrize("name", QUEUE_CASES)
def test_queue_and_candidate_boundaries(name, monkeypatch):
    """Slots with exactly N stage-1 survivors around the queue's capacity, real matches at queue indexes 0, 31, 32
    and N - 1 (the two-at-a-time judge, the 32-lane rounds); tiles with 1, 2, 3, 32 and 33 stage-2 survivors
    (pattern directory, sorted list, hand-over to the dense-match kernel)."""
    torch = torch_cuda()
    case = get_case(name)
    set_env(monkeypatch, case.spec)
    m = pf.Matcher(case.tables, device=0, n_streams=2, chunk_bytes=1 << 20)
    check_signature(m, case)
    text, tiles = queue_text(case)
    want = case.reference(text)
    assert len(want[0]) == sum(len({i for i in (0, 31, 32, n - 1) if i < n}) if kind == "queue" else n
                               for kind, n in tiles)
    d = torch.from_numpy(text).cuda()
    for _ in range(2):
        got = m.scan_device(d)
        check_launches(m, case)
        same(got, want, (name, "device"))
    same(m.scan_host(text), want, (name, "host"))
    m.close()
