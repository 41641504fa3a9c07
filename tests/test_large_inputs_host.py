"""Sparse references of the large-input tests (tests/test_large_inputs_gpu.py), and their CPU checks.

A scan of several GiB cannot be held to a full oracle scan, and it need not be: the texts are the background byte BG,
which no pattern contains, with clusters of other bytes planted at chosen positions.  A match cannot contain BG, so
the records of a range [a, b) are the union, over the clusters that meet it, of the reference's records of the
cluster clipped to [a, b), shifted to the cluster's place.  Patterns longer than 513 bytes meet the reference's
4096 + 512 walk bound (master_kernel.cu:141-144), which depends on where a start lies in the global 4096-byte grid
(base_pos + offset): such a cluster is scanned behind BG padding back to the previous global multiple of 4096, so
that the reference's tile phase equals the kernel's.

A flow's stream is modelled as a sequence of views of one such text: the records are the clusters inside each view
plus one reference scan per seam, over the last max_len - 1 bytes before it and the first max_len - 1 after it."""
import bisect

import numpy as np
import pytest

import phfpfac_b200 as pf
from _oracle import Oracle
from test_detector_paths_host import BG, REF_HALO, TILE, get_case, lines_of, phase_text

PAGE = 4096                       # the reference's tile (master_kernel.cu:9-10): grid of the walk bound
LARGE_CASES = ["A", "F", "F2", "H", "J1", "J3"]
FIN_THREADS = 256                 # kFinThreads: tiles the ordering pass moves per chunk of a CTA's range
MAX_PARTS = 1024                  # kMaxParts: CTAs of the ordering pass


def max_call_bytes(mis):
    """The largest n_valid a scan call accepts at pointer misalignment mis = d_in & 15.  launch_scan
    (pfac_device.cu) refuses min(n_valid, n_starts + M - 1) + mis + kTile + 4096 >= 2^32, which keeps the kernels'
    32-bit positions (tile starts, a_valid_end, record positions, the ring's prefetch) in range; the batch total and
    the packed bytes of a flow call are held to the same bound."""
    return 2 ** 32 - TILE - PAGE - 1 - mis


def ordering_ranges(n_starts, mis):
    """(n_tiles, tiles per CTA of the ordering pass) of a scan: launch_scan gives each pfac_finalize_kernel CTA
    ceil(n_tiles / fgrid) tiles, fgrid = min(ceil(n_tiles / 8), 1024), walked 256 at a time."""
    n_tiles = -(-(mis + n_starts) // TILE)
    fgrid = min(-(-n_tiles // 8), MAX_PARTS)
    return n_tiles, -(-n_tiles // fgrid)


# ---------------------------------------------------------------- plant layouts

class Plants:
    """Clusters of bytes at chosen positions of a text of background bytes, kept more than `gap` bytes apart (a
    cluster may hold background bytes of its own).  put() refuses a cluster that would come closer."""

    def __init__(self, gap, bg=BG):
        self.gap, self.bg = gap, bg
        self.starts, self.blobs = [], []

    def free(self, at, blob):
        i = bisect.bisect_left(self.starts, at)
        if i > 0 and self.starts[i - 1] + len(self.blobs[i - 1]) + self.gap >= at:
            return False
        return not (i < len(self.starts) and at + len(blob) + self.gap >= self.starts[i])

    def put(self, at, blob):
        blob = bytes(blob)
        if at < 0 or not blob or not self.free(at, blob):
            return False
        i = bisect.bisect_left(self.starts, at)
        self.starts.insert(i, at)
        self.blobs.insert(i, blob)
        return True

    def must_put(self, at, blob):
        assert self.put(at, blob), ("no room for a cluster at", at)

    def shifted(self, d):
        p = Plants(self.gap, self.bg)
        p.starts, p.blobs = [s + d for s in self.starts], list(self.blobs)
        return p

    def merged(self, other):
        """Both sets of clusters (they must not overlap); clusters that touch become one."""
        p = Plants(0, self.bg)
        for s, b in sorted(list(zip(self.starts, self.blobs)) + list(zip(other.starts, other.blobs))):
            if p.starts and p.starts[-1] + len(p.blobs[-1]) == s:
                p.blobs[-1] += b
            else:
                assert not p.starts or p.starts[-1] + len(p.blobs[-1]) < s
                p.starts.append(s)
                p.blobs.append(b)
        return p

    def __iter__(self):
        return iter(zip(self.starts, self.blobs))

    def meeting(self, a, b):
        """Clusters that meet [a, b)."""
        i = max(bisect.bisect_right(self.starts, a) - 1, 0)
        j = bisect.bisect_left(self.starts, b)
        return [(s, bl) for s, bl in zip(self.starts[i:j], self.blobs[i:j]) if s + len(bl) > a]

    def text(self, a, n):
        """The bytes [a, a + n) as a host array."""
        out = np.full(n, self.bg, dtype=np.uint8)
        for s, bl in self.meeting(a, a + n):
            lo, hi = max(s, a), min(s + len(bl), a + n)
            out[lo - a:hi - a] = np.frombuffer(bl, dtype=np.uint8)[lo - s:hi - s]
        return out


class Reference:
    """A reference scan `ref(array) -> (pos int64[], id int32[])` over texts whose background is `bg`; `paged`: the
    set has patterns longer than 513 bytes (the walk bound depends on the global 4096-byte grid).  The records of
    each (cluster piece, padding) are computed once."""

    def __init__(self, ref, bg=BG, paged=False):
        self.ref, self.bg, self.paged = ref, bg, paged
        self.cache = {}

    def piece(self, blob, pad):
        key = (blob, pad)
        if key not in self.cache:
            text = np.concatenate([np.full(pad, self.bg, dtype=np.uint8), np.frombuffer(blob, dtype=np.uint8)])
            pos, ids = self.ref(text)
            self.cache[key] = (pos - pad, ids)
        return self.cache[key]

    def __call__(self, plants, a, n_valid, n_starts=None, base_pos=0):
        """Records of a scan of text[a, a + n_valid) with starts below n_starts, positions relative to a; base_pos =
        global position of text[a]."""
        n_starts = n_valid if n_starts is None else n_starts
        P, I = [np.zeros(0, np.int64)], [np.zeros(0, np.int32)]
        for s, bl in plants.meeting(a, a + n_valid):
            lo, hi = max(s, a), min(s + len(bl), a + n_valid)
            rel = lo - a
            pad = (base_pos + rel) % PAGE if self.paged else 0
            pos, ids = self.piece(bl[lo - s:hi - s], pad)
            P.append(pos + rel)
            I.append(ids)
        pos, ids = np.concatenate(P), np.concatenate(I)
        keep = pos < n_starts
        return pos[keep], ids[keep]


def case_reference(case):
    if not hasattr(case, "_large_ref"):
        case._large_ref = Reference(case.reference, BG, case.max_len > REF_HALO + 1)
    return case._large_ref


def small_plants(case):
    """Patterns of at most 24 bytes (or the shortest ones): fillers of the layouts."""
    return [p for p in case.lines if len(p) <= 24][:400] or sorted(case.lines, key=len)[:400]


def straddler(case):
    """The longest pattern of at most 64 bytes: planted across the points where positions cross 2^31 or 2^32."""
    return max((p for p in case.lines if len(p) <= 64), key=len)


def phase_block(case):
    """The plants of phase_text (every plant at the lane, slice, slot and tile phases in tiles of 1, 2, 3-32 and more
    than 32 plants, near-misses) without its end zone, as one cluster that starts on a tile border."""
    if not hasattr(case, "_phase_block"):
        text, info = phase_text(case)
        body = text[:info["border"]]
        last = int(np.nonzero(body != BG)[0][-1]) + 1
        case._phase_block = body[:last].tobytes()
    return case._phase_block


def scan_layout(case, n, mis, mid=1 << 31, base_pos=0, straddle=1, block_at=None):
    """Clusters of one scan of n bytes at misalignment mis (positions relative to the call's first start; the kernel's
    tile grid is at pos + mis):
    - the straddler across `mid`, `straddle` bytes of it below;
    - the phase block past `mid` (or below it when the call ends too soon after it);
    - in the ordering pass's ranges of CTAs 0, 1, the middle and the last two: a plant in the first tile, in the
      first tile of the range's second 256-tile chunk (where the range has one) and in the last tile;
    - 900-byte plants around the walk-bound cut (global starts 3707-3710 past a multiple of 4096) where the set has
      them, and the longest pattern across tile borders near `mid`;
    - the end zone: the longest pattern starting on the last tile border it fits behind, and a pattern ending
      exactly at n (unless the straddler reaches n).
    Returns (plants, {"end": start of the pattern that ends at n or None, "border": ...})."""
    P = Plants(case.max_len)
    s = straddler(case)
    P.must_put(mid - straddle, s)
    fill = small_plants(case)
    block = phase_block(case)
    past = n >= mid + len(block) + (4 << 20)
    zone = mid + (64 << 10) if past else mid - (448 << 10)      # 384 KiB for the tile-border and walk-bound plants
    if block_at is None:
        if past:
            block_at = (mid + (1 << 20) + mis) // TILE * TILE - mis
        else:
            block_at = (mid - (512 << 10) - len(block) + mis) // TILE * TILE - mis
    P.must_put(block_at, block)
    n_tiles, per = ordering_ranges(n, mis)
    fgrid = -(-n_tiles // per)
    k = 0
    for b in sorted({0, 1, fgrid // 2, fgrid - 2, fgrid - 1}):
        for t in (b * per, b * per + FIN_THREADS, b * per + per - 1):
            if t >= min((b + 1) * per, n_tiles) or (t == b * per + FIN_THREADS and per <= FIN_THREADS):
                continue
            q = fill[(7 * k) % len(fill)]
            k += 1
            for r in (100, 1000, 3000, 5000, 7000):
                at = t * TILE + r + k % 13 - mis
                if at + len(q) <= n - 2 * case.max_len - 4 * TILE and P.put(at, q):
                    break
    longest = max(case.lines, key=len)
    if case.max_len > REF_HALO + 1:
        page = (base_pos + zone) // PAGE * PAGE
        for j, r in enumerate((3707, 3708, 3709, 3710)):
            P.must_put(page + (2 * j + 1) * 2 * PAGE + r - base_pos, longest)
    for j, d in enumerate((1, len(longest) // 2, len(longest) - 1)):
        P.must_put((zone + (256 << 10) + mis) // TILE * TILE + (2 * j + 1) * TILE - mis - d, longest)
    end_p = fill[len(fill) // 3]
    end = n - len(end_p)
    if not P.put(end, end_p):      # (the straddler already runs past n when n is just above `mid`)
        end = None
    border = (n - 2 * case.max_len - 2 * TILE + mis) // TILE * TILE - mis
    P.must_put(border, longest)
    return P, {"end": end, "end_len": len(end_p), "border": border}


class FlowCase:
    """Case A's set with one more line, "dex.html HTTP/1.1", so that "GET /index.html HTTP/1.1" cut after "GET /in"
    has a match ending at the cut ("GET /in"), one starting there (the new line) and two across it."""
    EXTRA = b"dex.html HTTP/1.1\n"

    def __init__(self):
        base = get_case("A")
        self.name, self.spec = "A+", base.spec
        self.blob = base.blob + self.EXTRA
        self.lines = lines_of(self.blob)
        assert len(set(self.lines)) == len(self.lines) and all(BG not in p for p in self.lines)
        self.lens = np.array([len(p) for p in self.lines], dtype=np.int64)
        self.max_len, self.min_len = int(self.lens.max()), int(self.lens.min())
        self.tables = pf.Tables.from_bytes(self.blob, 1, 256)
        self._oracle = Oracle(self.blob, 1, 256)

    def reference(self, data):
        return self._oracle.scan(np.ascontiguousarray(data, dtype=np.uint8))


_FLOW_CASE = []


def flow_case():
    if not _FLOW_CASE:
        _FLOW_CASE.append(FlowCase())
    return _FLOW_CASE[0]


def seam_split(case):
    """(S, j): a pattern S of at most 64 bytes and a cut j such that another pattern ends at j and one starts at j;
    a stream whose chunk ends with S[:j] and whose next chunk starts with S[j:] has a straddling match (S), a match
    ending at the seam and one starting there.  None if the set has none."""
    ref = case.reference
    for S in sorted((p for p in case.lines if len(p) <= 64), key=lambda p: (-len(p), p)):
        pos, ids = ref(np.frombuffer(S, dtype=np.uint8))
        end = pos + case.lens[ids - 1]
        for j in range(1, len(S)):
            if (end == j).any() and (pos == j).any():
                return S, j
    return None


def flow_view(case, c, split, inner=()):
    """Clusters of one view of c bytes: S[j:] at its start and S[:j] at its end (split = (S, j)), so that every seam
    between two views carries S; small plants at the offsets `inner`."""
    S, j = split
    P = Plants(case.max_len)
    P.must_put(0, S[j:])
    P.must_put(c - j, S[:j])
    fill = small_plants(case)
    for k, at in enumerate(inner):
        P.must_put(at, fill[(5 * k + 1) % len(fill)])
    return P


def stream_reference(case, plants, views):
    """Records (stream positions, in (pos, pattern length) order) of a flow whose stream is the views [(start,
    length)] of the text `plants` describes: each view's own clusters, plus what crosses each seam."""
    ref = case_reference(case)
    M1 = case.max_len - 1
    P, I = [np.zeros(0, np.int64)], [np.zeros(0, np.int32)]
    at = 0
    for k, (s, c) in enumerate(views):
        pos, ids = ref(plants, s, c)
        P.append(pos + at)
        I.append(ids)
        if k > 0:
            ps, pc = views[k - 1]
            assert pc >= M1
            window = np.concatenate([plants.text(ps + pc - M1, M1), plants.text(s, min(M1, c))])
            pos, ids = case.reference(window)
            keep = (pos < M1) & (pos + case.lens[ids - 1] > M1)
            P.append(pos[keep] + at - M1)
            I.append(ids[keep])
        at += c
    pos, ids = np.concatenate(P), np.concatenate(I)
    order = np.lexsort((case.lens[ids - 1], pos))
    return pos[order], ids[order]


# ---------------------------------------------------------------- CPU tests

def test_max_call_bytes_is_the_guard_of_launch_scan():
    import os
    src = open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "phfpfac_b200", "csrc",
                            "pfac_device.cu")).read()
    assert "n_valid + mis + (uint64_t)kTile + 4096 >= (1ull << 32)" in src
    assert "packed + (uint64_t)kTile + 4096 >= (1ull << 32)" in src
    assert max_call_bytes(0) + 0 + TILE + PAGE == 2 ** 32 - 1 and max_call_bytes(15) == 2 ** 32 - 12289 - 15
    assert ordering_ranges(1 << 31, 0) == (262144, 256) and ordering_ranges((1 << 31) + 1, 0)[1] == 257
    assert ordering_ranges(max_call_bytes(15), 15) == (524287, 512)


@pytest.mark.parametrize("name", LARGE_CASES)
def test_sparse_reference_equals_the_whole_text_scan(name):
    """The same plant classes as the GPU layouts, gaps shrunk (2^31 -> 3 MiB, n = 18 MiB): the sparse reference equals
    the reference's scan of the whole text, for whole calls, shifted ones, cut ones and n_starts < n_valid."""
    case = get_case(name)
    ref = case_reference(case)
    n, mid = 18 << 20, 3 << 20
    for mis, straddle in ((0, 1), (15, len(straddler(case)) - 1)):
        P, info = scan_layout(case, n, mis, mid=mid, straddle=straddle)
        text = P.text(0, n + 4096)
        want = case.reference(text[:n])
        got = ref(P, 0, n)
        assert len(want[0]) > 100 and np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (name, mis)
        wend = want[0] + case.lens[want[1] - 1]
        for a, nv, ns in ((mid - 5, n - mid + 5, None), (0, n - 1, None), (0, n, info["end"]), (0, n, info["end"] + 1),
                          (info["border"] - 7, 4096, 3)):
            ns_ = nv if ns is None else ns
            if case.max_len > REF_HALO + 1:
                wp, wi = case.reference(text[a:a + nv])
            else:   # a match is reported iff it lies inside the range
                keep = (want[0] >= a) & (wend <= a + nv)
                wp, wi = want[0][keep] - a, want[1][keep]
            keep = wp < ns_
            got = ref(P, a, nv, ns)
            assert np.array_equal(got[0], wp[keep]) and np.array_equal(got[1], wi[keep]), (name, mis, a, nv, ns)
    if case.max_len > REF_HALO + 1:
        # a call whose first byte lies at a global position that is a multiple of 4096 (the tile phase is the
        # whole text's), and one at 1234 past such a multiple (the text behind that many background bytes)
        P, _ = scan_layout(case, n, 0, mid=mid, base_pos=3 * PAGE)
        text = P.text(0, n)
        want = case.reference(text)
        got = ref(P, 0, n, base_pos=3 * PAGE)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
        bp = (1 << 32) + 4096 * 5 + 1234
        P, _ = scan_layout(case, n, 0, mid=mid, base_pos=bp)
        text = P.text(0, n)
        want = case.reference(np.concatenate([np.full(bp % PAGE, BG, dtype=np.uint8), text]))
        got = ref(P, 0, n, base_pos=bp)
        assert np.array_equal(got[0], want[0] - bp % PAGE) and np.array_equal(got[1], want[1])
        # the walk-bound plants: the reference keeps the 900-byte ones up to 3708 past a page and cuts the others
        L = case.max_len
        starts = got[0][case.lens[got[1] - 1] == L] + bp
        assert {3707, 3708} <= set((starts % PAGE).tolist()) and not {3709, 3710} & set((starts % PAGE).tolist())


def test_flow_stream_model_equals_the_whole_stream_scan():
    """The stream model of the flow tests, with 64 KiB views instead of 1 GiB ones, equals the reference's scan of the
    concatenated stream: per-view clusters plus one scan per seam."""
    case = flow_case()
    split = seam_split(case)
    assert split is not None
    c = 64 << 10
    views_p = [flow_view(case, c, split, (1000, 30000)), flow_view(case, c - 123, split, (777,)),
               flow_view(case, c + 4097, split, ())]
    for V in views_p:
        P = V.shifted(5)
        last = max(s + len(b) for s, b in P)
        c_ = last - 5
        for n_views in (1, 2, 5):
            views = [(5, c_)] * n_views
            stream = np.concatenate([P.text(5, c_)] * n_views)
            want = case.reference(stream)
            order = np.lexsort((case.lens[want[1] - 1], want[0]))
            got = stream_reference(case, P, views)
            assert np.array_equal(got[0], want[0][order]) and np.array_equal(got[1], want[1][order])
            if n_views > 1:   # the seams carry S, and matches end and start on them
                S, j = split
                ends = got[0] + case.lens[got[1] - 1]
                for k in range(1, n_views):
                    assert ((got[0] == k * c_ - j) & (case.lens[got[1] - 1] == len(S))).any()
                    assert (ends == k * c_).any() and (got[0] == k * c_).any()
    # views of different lengths and places
    P = views_p[0].merged(views_p[1].shifted(c + 50))
    views = [(0, c), (c + 50, c - 123), (0, c), (0, 70000)]
    stream = np.concatenate([P.text(s, n) for s, n in views])
    want = case.reference(stream)
    order = np.lexsort((case.lens[want[1] - 1], want[0]))
    got = stream_reference(case, P, views)
    assert np.array_equal(got[0], want[0][order]) and np.array_equal(got[1], want[1][order])
