"""Pattern sets, texts and references of the detector-path tests (tests/test_detector_paths_gpu.py), and their
CPU checks: the brute-force reference equals the oracle, the background byte has no stage-1 survivor, every
queue text hits its survivor count in the host model of the filters, and the tile geometry the texts are laid
out against is the geometry of pfac_kernel.cuh.

A scan runs one of several detector kernels (pfac_device.cu, detector_kernel), chosen by the derived tables
(pfac_derive.cc, derive_tables) and pfac_ctx_create.  Each case below is a pattern set, an environment and the
signature the GPU test asserts, so that a case that drifts off its kernel fails instead of passing with less
coverage.  Texts are a background byte that no pattern contains, with patterns planted at controlled
tile-relative phases."""
import os
import re
from functools import lru_cache

import numpy as np
import pytest

import phfpfac_b200 as pf
import pfac_synth as synth
from _oracle import Oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNEL_H = os.path.join(ROOT, "phfpfac_b200", "csrc", "pfac_kernel.cuh")

# tile geometry of the detector (pfac_kernel.cuh; test_kernel_constants_match_the_header checks it)
SLICE = 512                             # kSlice: starts per stage-1 step of a warp (32 lanes x 16 B)
TILE_SLICES = 16                        # PFAC_TILE_SLICES
TILE = SLICE * TILE_SLICES              # 8,192 starts per tile
LANE = 16
SLOT_SLICES = {0: 4, 1: 2, 2: 4}        # PFAC_SLOT_SLICES2 (mode 0), PFAC_SLOT_SLICES (mode 1), PFAC_SLOT_SLICES_GLOBAL
Q1_CAP = {m: 64 * s for m, s in SLOT_SLICES.items()}   # stage-1 queue of a slot; more survivors: the tile goes whole
CAND_PER_TILE = 32                      # kCandPerTile
DIR_CAND = 2                            # kDirCand: tiles with at most this many candidates probe the directory
REF_HALO = 512                          # patterns longer than 513 B meet the reference's 4096 + 512 walk bound
T2_GLOBAL_BYTES = 131072                # T2 of global mode after pfac_ctx_create widens it

BG = 10                                 # background byte: '\n' cannot be inside a pattern
NESTED = b"GET /index\nGET /in\nGET /index.html HTTP/1.1\n"


def lines_of(blob):
    return blob.split(b"\n")[:-1]


def _rand_pat(rng, n):
    p = rng.integers(0, 256, n).astype(np.uint8)
    p[p == BG] = BG + 1
    return p.tobytes()


def snort_like(shortest, seed):
    """Every length from `shortest` to `shortest` + 4 and a longer tail, plus prefix-sharing groups: one 4-byte prefix,
    a member of the shortest length (m1 of the prefix), members that share it and go on (m1 < len) and members that
    leave it at byte m1 - 4 .. m1 - 1 (a level-2 group with m2 > m1)."""
    rng = np.random.default_rng(seed)
    pats = []
    for i in range(1500):
        L = shortest + i % 5 if i < 1200 else int(rng.integers(shortest, 41))
        pats.append(_rand_pat(rng, L))
    for g in range(80):
        p4 = _rand_pat(rng, 4)
        short = p4 + _rand_pat(rng, shortest - 4)
        other = p4 + _rand_pat(rng, shortest - 4)
        pats += [short, short + _rand_pat(rng, 5), short + _rand_pat(rng, 20), other + _rand_pat(rng, 3),
                 other + _rand_pat(rng, 8), p4 + _rand_pat(rng, shortest + 8)]
    seen, out = set(), []
    for p in pats:
        if p not in seen:
            seen.add(p)
            out.append(p)
    return b"".join(p + b"\n" for p in out)


def long_tail(lengths, seed):
    rng = np.random.default_rng(seed)
    return b"".join(_rand_pat(rng, L) + b"\n" for L in lengths)


# queue texts: runs of QP's first two bytes, repeated, give stage-1 survivors (how many per run length: run_lengths)
# and no match (QP goes on differently); RP is a short real pattern with one survivor.  Both join the case sets.
QP_TAIL = b"\x7f\x7e\x7d\x7c"
RP = {6: b"\x11\x22\x33\x44\x55\x66", 7: b"\x11\x22\x33\x44\x55\x66\x77"}
QP_PAIRS = [(1, 2), (3, 4), (5, 6), (7, 8), (0x21, 0x43), (0x65, 0x87), (0xa9, 0xcb)]


def queue_extras(shortest, pair):
    a, b = pair
    return bytes([a, b] * 3) + QP_TAIL + b"\n" + RP[7 if shortest >= 7 else 6] + b"\n"


@lru_cache(maxsize=None)
def base_blob(name):
    if name == "A":
        return synth.synth_patterns(1, 3000, 3, 4, 64) + NESTED
    if name.startswith("C"):
        return snort_like(int(name[1:]), 40 + int(name[1:]))
    if name == "H":
        return synth.synth_patterns(1, 30000, 7, 4, 12)
    if name == "I":
        return synth.synth_patterns(0, 30000, 5, 8, 32)
    raise KeyError(name)


# name -> base set, extra patterns, environment, expected signature.  kernel: what a scan of it runs
# (pfac_device.cu, detector_kernel; or the dense-match kernel alone)
# (T/F = HAS_SHORT, HAS_SC, W3 of pfac_scan2_kernel).  launches: 3 = detector + dense-match + ordering pass,
# 1 = the dense-match kernel alone (DIRECT).  ref: "oracle" (Oracle, one partition), "brute" (brute_force) or
# "tables" (the oracle's scan over the case's own canonical arrays).
CASES = {
    "A": dict(base="A", env={}, kernel="pfac_scan2_kernel<F,T,T>", mode=0, has_short=0, level2=True, launches=3, shortest=4, queue=True),
    "B": dict(base="A", env={"PFAC_NO_W3": "1"}, kernel="pfac_scan2_kernel<F,T,F>", mode=0, has_short=0, level2=True, launches=3, shortest=4),
    "C5": dict(base="C5", env={}, kernel="pfac_scan2_kernel<F,F,T>", mode=0, has_short=0, level2=True, launches=3, shortest=5, queue=True),
    "C6": dict(base="C6", env={}, kernel="pfac_scan2_kernel<F,F,T>", mode=0, has_short=0, level2=True, launches=3, shortest=6, queue=True),
    "C7": dict(base="C7", env={}, kernel="pfac_scan2_kernel<F,F,T>", mode=0, has_short=0, level2=True, launches=3, shortest=7, queue=True),
    "D5": dict(base="C5", env={"PFAC_NO_W3": "1"}, kernel="pfac_scan2_kernel<F,F,F>", mode=0, has_short=0, level2=True, launches=3, shortest=5),
    "D6": dict(base="C6", env={"PFAC_NO_W3": "1"}, kernel="pfac_scan2_kernel<F,F,F>", mode=0, has_short=0, level2=True, launches=3, shortest=6),
    "D7": dict(base="C7", env={"PFAC_NO_W3": "1"}, kernel="pfac_scan2_kernel<F,F,F>", mode=0, has_short=0, level2=True, launches=3, shortest=7),
    "E": dict(base="A", env={"PFAC_TM2_BYTES": "0"}, kernel="pfac_scan2_kernel<F,T,T> without level 2", mode=0, has_short=0, level2=False, launches=3, shortest=4),
    "F": dict(base="A", extra=("long", (100, 150, 200)), env={}, kernel="pfac_scan2_kernel<F,T,T>, no pattern directory", mode=0, has_short=0, level2=True, launches=3, shortest=4, max_len=200),
    "F2": dict(base="A", extra=("long", (600, 900)), env={}, kernel="pfac_scan2_kernel<F,T,T>, reference tile bound", mode=0, has_short=0, level2=True, launches=3, shortest=4, max_len=900),
    "G": dict(base="A", dag=True, env={}, kernel="pfac_scan2_kernel<F,T,T> on a DAG", mode=0, has_short=0, level2=True, launches=3, shortest=4, ref="tables"),
    "H": dict(base="H", env={}, kernel="pfac_scan_kernel<2>", mode=2, has_short=0, level2=True, launches=3, shortest=4, ref="brute", queue=True),
    "I": dict(base="I", env={}, kernel="pfac_scan_kernel<2>", mode=2, has_short=0, level2=True, launches=3, shortest=8, ref="brute", no_rp=True),
    "J1": dict(base="H", extra=("raw", b"ab\n"), env={"PFAC_DENSE_FIRST": "0"}, kernel="pfac_scan_kernel<1>", mode=1, has_short=1, level2=False, launches=3, shortest=2, ref="brute", queue=True),
    "J2": dict(base="A", extra=("raw", b"ab\n"), env={"PFAC_DENSE_FIRST": "0"}, kernel="pfac_scan2_kernel<T,T,F>", mode=0, has_short=1, level2=True, launches=3, shortest=2),
    "J3": dict(base="A", env={"PFAC_DENSE_FIRST": "1"}, kernel="pfac_dense_kernel<true> alone", mode=0, has_short=0, level2=True, launches=1, shortest=4),
}
QUEUE_CASES = [k for k, v in CASES.items() if v.get("queue")]


def queue_counts(mode):
    cap = Q1_CAP[mode]
    return [1, 31, 32, 33, 63, 64, 65, cap - 1, cap, cap + 1]


def set_env(monkeypatch, case):
    for k in ("PFAC_NO_W3", "PFAC_TM2_BYTES", "PFAC_DENSE_FIRST"):
        monkeypatch.delenv(k, raising=False)
    for k, v in case["env"].items():
        monkeypatch.setenv(k, v)


def profile_bytes(case):
    """t2_bytes of the stage-1 model: global mode's stage 1 is T2 at the size the device widens it to."""
    return T2_GLOBAL_BYTES if case.spec["mode"] == 2 else 32768


class Case:
    """The pattern set of a case, its tables and its reference scan."""

    def __init__(self, name, qp_pair=(1, 2)):
        c = self.spec = CASES[name]
        self.name = name
        blob = base_blob(c["base"])
        kind, extra = c.get("extra", (None, None))
        if kind == "long":
            blob += long_tail(extra, 77)
        elif kind == "raw":
            blob += extra
        if not c.get("no_rp"):
            blob += queue_extras(c["shortest"], qp_pair)
        else:
            blob += bytes([qp_pair[0], qp_pair[1]] * 3) + QP_TAIL + b"\n"
        self.qp_pair = qp_pair
        self.blob = blob
        self.lines = lines_of(blob)
        assert len(set(self.lines)) == len(self.lines) and all(BG not in p for p in self.lines)
        self.lens = np.array([len(p) for p in self.lines], dtype=np.int64)
        self.tables = pf.Tables.from_bytes(blob, 1, 256)
        if c.get("dag"):
            p = self.tables.part(0)
            s0 = p.s0.copy()
            used = {q[0] for q in self.lines}
            self.dag_bytes = {}
            donors = sorted({q[0] for q in self.lines if len(q) >= 6})
            for k, b in enumerate(sorted(set(range(256)) - used - {BG})):
                s0[b] = s0[donors[(7 * k) % len(donors)]]     # a second root edge into an existing first state
                self.dag_bytes[b] = donors[(7 * k) % len(donors)]
            assert self.dag_bytes
            self.tables = pf.Tables.from_arrays(s0, p.r, p.HT, p.val, 256, p.state_num, p.n_final, p.idmap, p.max_len)
            self.part = self.tables.part(0)
        self.max_len = int(self.lens.max())
        self.min_len = int(self.lens.min())
        self.rp = RP[7 if c["shortest"] >= 7 else 6]
        self._oracle = None

    # ---- reference scans
    def reference(self, data):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        ref = self.spec.get("ref", "oracle")
        if ref == "brute":
            return brute_force(self.lines, data)
        if ref == "tables":
            from _oracle import scan_tables_cpu
            return scan_tables_cpu(self.part, self.part.idmap, self.max_len, data)
        if self._oracle is None:
            self._oracle = Oracle(self.blob, 1, 256)
        return self._oracle.scan(data)

    # ---- pattern roles of the phase texts
    def m1(self, p):
        return int(min([len(q) for q in self.lines if q[:4] == p[:4]] or [len(p)]))

    def plants(self):
        """shortest, one of each length from the shortest to shortest + 4, longest, nested, a member with m1 < len."""
        L = self.lines
        by_len = {}
        for p in L:
            by_len.setdefault(len(p), p)
        out = [min(L, key=len)]
        out += [by_len[k] for k in range(self.min_len, self.min_len + 5) if k in by_len and by_len[k] not in out]
        out.append(max(L, key=len))
        lset = set(L)
        nested = [p for p in L if len(p) > 4 and any(p[:k] in lset for k in range(1, len(p)))]
        if nested:
            out.append(max(nested, key=lambda p: sum(p[:k] in lset for k in range(1, len(p)))))
        heads = {}
        for p in L:
            if len(p) >= 4:
                heads[p[:4]] = min(heads.get(p[:4], 1 << 30), len(p))
        grouped = [p for p in L if len(p) >= 4 and heads[p[:4]] < len(p) <= 64]
        if grouped:
            out.append(grouped[len(grouped) // 2])
        if self.spec.get("dag"):   # a start through a redirected root edge
            b, donor = next(iter(self.dag_bytes.items()))
            src = next(p for p in L if p[0] == donor and len(p) >= 6)
            out.append(bytes([b]) + src[1:])
        return out


@lru_cache(maxsize=None)
def get_case(name):
    """The case; for the queue cases, with the first queue pattern whose runs give 1..4 stage-1 survivors."""
    if not CASES[name].get("queue"):
        return Case(name)
    for pair in QP_PAIRS:
        case = Case(name, pair)
        case.runs = run_lengths(case)
        if case.runs:
            return case
    raise AssertionError(f"{name}: no queue pattern with a clean run")


def with_env(case_spec, fn):
    """Run fn() with the case's environment (the host model reads PFAC_NO_W3 when it derives the tables)."""
    saved = {k: os.environ.get(k) for k in ("PFAC_NO_W3", "PFAC_TM2_BYTES", "PFAC_DENSE_FIRST")}
    try:
        for k in saved:
            os.environ.pop(k, None)
        os.environ.update(case_spec["env"])
        return fn()
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def t1_pass(case, text):
    return with_env(case.spec, lambda: case.tables.filter_profile(text, 0, profile_bytes(case))["t1_pass"])


def to_emit(case, text):
    return with_env(case.spec, lambda: case.tables.filter_profile(text, 0, profile_bytes(case))["to_emit"])


# ---------------------------------------------------------------- brute force reference

def brute_force(lines, text):
    """Every (position, pattern) with text[pos:pos+len] == pattern, found by comparing windows of each distinct
    pattern length with the patterns of that length and verifying every hit byte by byte -- no automaton.
    Records in (position, pattern length) order; ids are 1-based line numbers (the set has no duplicates).  It
    knows nothing of the reference's 4096 + 512 walk bound: patterns of at most 513 bytes only."""
    assert len(set(lines)) == len(lines) and max(map(len, lines)) <= REF_HALO + 1
    text = np.ascontiguousarray(text, dtype=np.uint8)
    n = len(text)
    tb = text.tobytes()
    by_len = {}
    for i, p in enumerate(lines):
        by_len.setdefault(len(p), {})[p] = i + 1
    pad = np.concatenate([text, np.zeros(8, dtype=np.uint8)]).astype(np.uint64)
    key8 = np.zeros(n, dtype=np.uint64)
    for j in range(8):
        key8 |= pad[j:j + n] << np.uint64(8 * j)
    recs = []
    for L, d in by_len.items():
        if L > n:
            continue
        k = min(L, 8)
        mask = np.uint64((1 << (8 * k)) - 1)
        keys = np.unique(np.array([int.from_bytes(p[:k], "little") for p in d], dtype=np.uint64))
        win = key8[:n - L + 1] & mask
        idx = np.searchsorted(keys, win)
        idx[idx == len(keys)] = 0
        for i in np.nonzero(keys[idx] == win)[0].tolist():
            pid = d.get(tb[i:i + L])
            if pid is not None and all(tb[i + j] == lines[pid - 1][j] for j in range(L)):
                recs.append((i, L, pid))
    recs.sort()
    return (np.array([r[0] for r in recs], dtype=np.int64), np.array([r[2] for r in recs], dtype=np.int32))


# ---------------------------------------------------------------- texts with controlled phases

def phase_starts(mode):
    slot = SLOT_SLICES[mode] * SLICE
    return (list(range(0, 48)) + list(range(496, 528)) + list(range(slot - 16, slot + 16)) +
            list(range(TILE - 32, TILE)))


def near_misses(case, p):
    """Copies of p with one byte changed at index 0, 1, 3, 4, m1 - 1 or len - 1, and p without its last byte."""
    out = []
    for i in sorted({0, 1, 3, 4, case.m1(p) - 1, len(p) - 1}):
        if 0 <= i < len(p):
            q = bytearray(p)
            q[i] = (q[i] + 1) % 256
            if q[i] == BG:
                q[i] = BG + 1
            out.append(bytes(q))
    out.append(p[:-1])
    return out


class Layout:
    def __init__(self, n_tiles):
        self.text = np.full(n_tiles * TILE, BG, dtype=np.uint8)
        self.busy = np.zeros(n_tiles * TILE, dtype=bool)
        self.tile = 1                                  # tile 0 stays empty: the tiles below are interior ones

    def free(self, at, p, gap=1):
        return at >= 0 and at + len(p) + gap <= len(self.text) and not self.busy[max(0, at - gap):at + len(p) + gap].any()

    def put(self, at, p):
        self.text[at:at + len(p)] = np.frombuffer(p, dtype=np.uint8)
        self.busy[at:at + len(p)] = True

    def next_tile(self):
        while self.busy[self.tile * TILE:(self.tile + 1) * TILE].any():
            self.tile += 1
        t = self.tile
        self.tile += 1
        return t


def phase_text(case, rng_seed=0):
    """Plants at tile-relative starts 0-47, 496-527, the slot border and 8160-8191, in four layouts: one plant per
    tile (one candidate: the pattern directory), two per tile, 3-32 per tile (sorted candidate list) and more than
    32 (the tile goes to the dense-match kernel); near-misses in tiles of their own; an end zone.  Returns the text
    and the positions of note: {"plants": [...], "border": tile border of the end-zone bound, "cut": start of a
    pattern cut by a prefix length}."""
    rng = np.random.default_rng(rng_seed)
    plants = case.plants()
    starts = phase_starts(case.spec["mode"])
    pool = [p for p in case.lines if len(p) <= 24][:400] or case.lines[:400]
    lay = Layout(2048)
    placed = []

    def controlled(p, r, extra):
        while True:
            t = lay.next_tile()
            at = t * TILE + r
            if lay.free(at, p):
                break
        lay.put(at, p)
        placed.append(at)
        k = tries = 0
        while k < extra and tries < 20 * extra + 50:
            tries += 1
            q = pool[int(rng.integers(0, len(pool)))]
            a = t * TILE + int(rng.integers(0, TILE - len(q)))
            if lay.free(a, q):
                lay.put(a, q)
                k += 1
        assert k == extra
    # every plant at every start, once: half of the pairs alone in a tile (layout 1), the other half spread over
    # layouts 2 (one more plant in the tile), 3 (2-31 more) and 4 (40 more)
    for i, p in enumerate(plants):
        for j, r in enumerate(starts):
            if (i + j) % 2 == 0:
                controlled(p, r, 0)
            else:
                controlled(p, r, (1, 2 + (i + j) % 30, 40)[(j // 2) % 3])
    for i, p in enumerate(plants):        # near-misses: the oracle says which still match
        for k, q in enumerate(near_misses(case, p)):
            controlled(q, starts[(7 * i + 3 * k) % len(starts)], 0)
    # end zone: the longest pattern starting on a tile border (prefix lengths put n - max_len at -1, 0, +1 from it),
    # then a pattern cut by a prefix length, then the shortest pattern ending the input
    longest = max(case.lines, key=len)
    t = lay.next_tile() + 1
    border = t * TILE
    lay.put(border, longest)
    cut_p = plants[min(2, len(plants) - 1)]
    cut = border + len(longest) + 3 * TILE // 2
    lay.put(cut, cut_p)
    shortest = min(case.lines, key=len)
    end = cut + len(cut_p) + 700
    lay.put(end - len(shortest), shortest)
    text = lay.text[:end].copy()
    assert len(text) <= 16 << 20
    return text, {"plants": placed, "border": border, "cut": cut, "cut_len": len(cut_p)}


# ---------------------------------------------------------------- queue texts

def run_lengths(case):
    """{k: length of a run of the queue pattern's first two bytes, repeated, that gives exactly k stage-1 survivors}
    for k = 1..4, from the host model of the case's stage 1 (runs of at most 12 bytes: a lane keeps 4 background
    bytes, so no start of it sees the next lane); None unless the real pattern RP gives exactly one survivor."""
    a, b = case.qp_pair
    runs = {}
    for run in range(4, 13):
        text = np.full(64, BG, dtype=np.uint8)
        text[16:16 + run] = np.array(([a, b] * 8)[:run], dtype=np.uint8)
        runs.setdefault(t1_pass(case, text), run)
    text = np.full(64, BG, dtype=np.uint8)
    text[16:16 + len(case.rp)] = np.frombuffer(case.rp, dtype=np.uint8)
    if t1_pass(case, text) != 1 or not all(k in runs for k in (1, 2, 3, 4)):
        return None
    return runs


def lane_order(mode):
    """Tile-relative starts of a slot's lanes in the order their survivors enter the warp's queue: lane by lane,
    and within a lane slice by slice (the compaction of pfac_scan2_kernel / pfac_scan_kernel)."""
    return [h * SLICE + l * LANE for l in range(32) for h in range(SLOT_SLICES[mode])]


def queue_tile(case, n, real_at):
    """The bytes of one slot with exactly n stage-1 survivors; the survivors at queue indexes
    `real_at` are starts of the real pattern RP, all others are QP runs that stage 2 rejects.  A lane holds RP or a
    run with k = 1..4 survivors (run_lengths); a lane's survivors stay in its queue place whatever their offsets."""
    mode = case.spec["mode"]
    a, b = case.qp_pair
    lanes = lane_order(mode)
    slot = np.full(SLOT_SLICES[mode] * SLICE, BG, dtype=np.uint8)
    real = sorted(set(i for i in real_at if i < n))
    units, q = [], 0                          # survivors per lane in queue order; "rp" = one real match
    for r in real + [n]:
        seg = r - q                           # QP survivors before the next real one, in lanes of at most 4
        lanes_needed = -(-seg // 4)
        units += [seg // lanes_needed + (1 if i < seg % lanes_needed else 0) for i in range(lanes_needed)]
        if r < n:
            units.append("rp")
        q = r + 1
    assert len(units) <= len(lanes), (case.name, n)
    for off, u in zip(lanes, units):
        if u == "rp":
            slot[off:off + len(case.rp)] = np.frombuffer(case.rp, dtype=np.uint8)
        else:
            run = case.runs[u]
            slot[off:off + run] = np.array(([a, b] * 8)[:run], dtype=np.uint8)
    return slot


def queue_text(case):
    """Tiles 1, 3, 5, ... each with one slot of exactly N stage-1 survivors (N from queue_counts) and real matches at
    queue indexes 0, 31, 32 and N - 1; then tiles with 1, 2, 3, 32 and 33 stage-2 survivors (RP copies)."""
    mode = case.spec["mode"]
    counts = queue_counts(mode)
    emits = [1, 2, 3, 32, 33]
    n_tiles = 2 * (len(counts) + len(emits)) + 2 + case.max_len // TILE
    text = np.full(n_tiles * TILE, BG, dtype=np.uint8)
    tiles = {}
    for i, n in enumerate(counts):
        t = 1 + 2 * i
        slot_no = i % (TILE_SLICES // SLOT_SLICES[mode])
        at = t * TILE + slot_no * SLOT_SLICES[mode] * SLICE
        s = queue_tile(case, n, [0, 31, 32, n - 1])
        text[at:at + len(s)] = s
        tiles[("queue", n)] = (at, len(s))
    for j, k in enumerate(emits):
        t = 1 + 2 * (len(counts) + j)
        step = (TILE - 64) // k
        for i in range(k):
            a = t * TILE + 16 * ((i * step) // 16) + (i % 2) * 8
            text[a:a + len(case.rp)] = np.frombuffer(case.rp, dtype=np.uint8)
        tiles[("emit", k)] = (t * TILE, TILE)
    return text, tiles


# ---------------------------------------------------------------- CPU tests

def test_kernel_constants_match_the_header():
    src = open(KERNEL_H).read()

    def define(name):
        return int(re.search(r"#define\s+%s\s+(\d+)" % name, src).group(1))

    def const(name):
        return int(re.search(r"constexpr\s+int\s+%s\s*=\s*(\d+)\s*;" % name, src).group(1))
    assert const("kSlice") == SLICE and define("PFAC_TILE_SLICES") == TILE_SLICES
    assert define("PFAC_SLOT_SLICES2") == SLOT_SLICES[0] and define("PFAC_SLOT_SLICES") == SLOT_SLICES[1]
    assert define("PFAC_SLOT_SLICES_GLOBAL") == SLOT_SLICES[2]
    assert const("kCandPerTile") == CAND_PER_TILE and const("kDirCand") == DIR_CAND
    cap = re.search(r"constexpr\s+int\s+q1_cap\(int mode\)\s*\{\s*return\s+(\d+)\s*\*\s*slot_slices\(mode\)", src)
    assert cap and all(int(cap.group(1)) * SLOT_SLICES[m] == Q1_CAP[m] for m in SLOT_SLICES)
    assert re.search(r"kTile = kSlicesPerTile \* kSlice;\s*//\s*8,192 start positions per tile", src)


@pytest.mark.parametrize("name", ["A", "C5", "C6", "C7", "F"])
def test_brute_force_equals_the_oracle(name):
    case = get_case(name)
    text, _ = phase_text(case)
    text = text[:3 << 20]
    o = Oracle(case.blob, 1, 256)
    pos, ids = o.scan(text)
    bp, bi = brute_force(case.lines, text)
    assert len(pos) > 1000
    assert np.array_equal(bp, pos) and np.array_equal(bi, ids)


@pytest.mark.parametrize("name", list(CASES))
def test_background_has_no_stage1_survivor(name):
    case = get_case(name)
    bg = np.full(1 << 16, BG, dtype=np.uint8)
    assert t1_pass(case, bg) == 0
    assert len(case.reference(bg)[0]) == 0


@pytest.mark.parametrize("name", QUEUE_CASES)
def test_queue_texts_hit_their_counts(name):
    """Each queue slot has exactly N stage-1 survivors in the host model (modes 0 and 1: T1, independent of the
    shared-memory budgets; mode 2: T2 at the size the device widens it to); the emit tiles exactly k stage-2
    survivors."""
    case = get_case(name)
    text, tiles = queue_text(case)
    assert t1_pass(case, text) == sum(n for (kind, n) in tiles if kind == "queue") + sum(
        n for (kind, n) in tiles if kind == "emit")
    for (kind, n), (at, size) in tiles.items():
        window = text[at - 16:at + size + 16]
        if kind == "queue":
            assert t1_pass(case, window) == n, (kind, n)
            pos, ids = case.reference(window)
            assert len(pos) == len({i for i in (0, 31, 32, n - 1) if i < n}), n
        else:
            assert to_emit(case, window) == n and len(case.reference(window)[0]) == n, (kind, n)
