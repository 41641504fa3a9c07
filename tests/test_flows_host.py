"""Streaming scan of many flows (pfac_flows_*, Matcher.flows): a host model of the carry rule the device applies,
held to the oracle's scan of whole streams, and the ABI surface.  No GPU.

The rule (include/pfac_b200.h, DESIGN.md §3.9): a flow that has consumed P bytes carries its last
t = min(M - 1, P) bytes; the next chunk of c bytes is scanned as the document tail ++ chunk, and a record (p, L) of
that document is kept iff t < p + L <= t + c, at stream position P - t + p."""
import os
import re

import numpy as np
import pytest

import phfpfac_b200 as pf
from _oracle import Oracle
from phfpfac_b200._lib import ABI_SYMBOLS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLOW_SYMBOLS = ["pfac_flows_create", "pfac_flows_destroy", "pfac_flows_reset", "pfac_flows_position",
                "pfac_scan_flows_device_sync"]


def keep_rule(pos, ends, t, c):
    """Records of one document tail ++ chunk (t carried bytes, c new ones) that belong to the chunk."""
    return (ends > t) & (ends <= t + c)


def sort_records(pos, ids, lengths):
    order = np.lexsort((lengths[ids], pos))
    return pos[order], ids[order]


def model_stream(scan, lengths, M, chunks):
    """The records a flow gets, call by call, for `chunks` under the carry rule: [(pos int64[], id int32[])] with
    stream positions; scan(doc) -> (pos, id) of one document."""
    tail = np.zeros(0, dtype=np.uint8)
    P = 0
    out = []
    for ch in chunks:
        ch = np.asarray(ch, dtype=np.uint8)
        t = len(tail)
        assert t == min(M - 1, P)
        doc = np.concatenate([tail, ch])
        pos, ids = scan(doc)
        keep = keep_rule(pos, pos + lengths[ids], t, len(ch))
        out.append((pos[keep] + (P - t), ids[keep]))
        P += len(ch)
        tail = doc[len(doc) - min(M - 1, len(doc)):] if M > 1 else doc[:0]
    return out


def union(records, lengths):
    pos = np.concatenate([r[0] for r in records]) if records else np.zeros(0, dtype=np.int64)
    ids = np.concatenate([r[1] for r in records]) if records else np.zeros(0, dtype=np.int32)
    return sort_records(pos.astype(np.int64), ids.astype(np.int32), lengths)


def random_set(rng, alpha, n_pat, max_len):
    pats = set()
    for _ in range(50 * n_pat):
        if len(pats) >= n_pat:
            break
        L = int(rng.integers(1, max_len + 1))
        p = bytes(rng.integers(0, alpha, L).astype(np.uint8))
        if b"\n" not in p:
            pats.add(p)
    return b"".join(p + b"\n" for p in sorted(pats))


def special_sizes(M, shortest):
    """Chunk sizes at the carry's edges: empty, one byte, shorter than the shortest pattern, M - 2, M - 1, M."""
    return [0, 1, max(shortest - 1, 0), max(M - 2, 0), max(M - 1, 0), M]


def cut_stream(rng, text, sizes_pool, n):
    sizes = [int(sizes_pool[int(rng.integers(0, len(sizes_pool)))]) if rng.random() < 0.5
             else int(rng.integers(0, 3 * max(sizes_pool) + 2)) for _ in range(n)]
    chunks, at = [], 0
    for s in sizes:
        chunks.append(text[at:at + s])
        at += s
    return chunks, text[:at]


@pytest.mark.parametrize("seed", range(8))
def test_carry_rule_model_equals_whole_stream_scan(seed):
    rng = np.random.default_rng(500 + seed)
    alpha = [2, 3, 4, 8, 26, 3, 2, 5][seed]
    max_len = [4, 9, 20, 40, 12, 1, 70, 30][seed]
    blob = random_set(rng, alpha, int(rng.integers(1, 300)), max_len)
    t = pf.Tables.from_bytes(blob, 1, 256)
    lengths = t.pattern_lengths().astype(np.int64)
    M = t.max_pat_len
    shortest = min(len(p) for p in blob.split(b"\n")[:-1])
    o = Oracle(blob, 1, 256)
    text = rng.integers(0, alpha, 60000).astype(np.uint8)
    chunks, stream = cut_stream(rng, text, special_sizes(M, shortest), 120)
    got = model_stream(o.scan, lengths, M, chunks)
    want = sort_records(*[np.asarray(x) for x in o.scan(stream)], lengths)
    u = union(got, lengths)
    assert len(u[0]) == len(want[0]) and np.array_equal(u[0], want[0]) and np.array_equal(u[1], want[1])
    # every record ends in its own chunk, and within a chunk records are ordered by (pos, pattern length)
    P = 0
    for ch, (pos, ids) in zip(chunks, got):
        ends = pos + lengths[ids]
        assert ((ends > P) & (ends <= P + len(ch))).all()
        key = list(zip(pos.tolist(), lengths[ids].tolist()))
        assert key == sorted(key)
        P += len(ch)


def test_carry_rule_straddles_and_reports_once():
    """'nee|dle' across two chunks is reported once, in the chunk where it ends; a match ending exactly at a chunk's
    end is reported in that call and never again."""
    blob = b"needle\nle\nhaystack\n"
    t = pf.Tables.from_bytes(blob, 1, 256)
    lengths = t.pattern_lengths().astype(np.int64)
    o = Oracle(blob, 1, 256)
    chunks = [np.frombuffer(c, dtype=np.uint8) for c in (b"xxnee", b"dlexxneedle", b"", b"hay", b"stack")]
    got = model_stream(o.scan, lengths, t.max_pat_len, chunks)
    assert [len(p) for p, _ in got] == [0, 4, 0, 0, 1]
    assert got[1][0].tolist() == [2, 6, 10, 14] and got[4][0].tolist() == [16]


def test_header_declares_the_flow_symbols():
    src = open(os.path.join(ROOT, "include", "pfac_b200.h")).read()
    code = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    for name in FLOW_SYMBOLS:
        assert re.search(r"\b%s\s*\(" % name, code), name
        assert name in ABI_SYMBOLS, name
    assert "typedef struct pfac_flows pfac_flows;" in code
    assert pf.FLOW_MATCH_DTYPE.names == ("pos", "id") and pf.FLOW_MATCH_DTYPE["pos"] == np.dtype("<u8")
