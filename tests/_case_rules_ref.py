"""Reference for pattern sets with per-pattern case rules (PFAC_PATTERNS_CASE_RULES), built on the unchanged oracle
(tests/_oracle.py) like tests/_caseless_ref.py.

rules[i] = 1: pattern id i + 1 matches where fold(T[pos, pos+L)) == fold(p); 0: where T[pos, pos+L) == p.  Duplicates
are decided within a rule class (the last line wins), so the reference is two oracle runs:
  1. the caseless lines, folded, over fold(T);
  2. the exact lines over T;
their sub-file ids mapped back to line numbers, and the two record sets merged by (pos, length, id).  With escapes
the patterns are decoded and each sub-file is written back as octal escapes (decode_escapes, octal_file)."""
import numpy as np

from _caseless_ref import decode_escapes, fold, octal_file
from _oracle import Oracle


def patterns_of(blob, escapes=False):
    """The patterns the reader returns, in file order."""
    if escapes:
        return decode_escapes(blob)
    assert blob.endswith(b"\n")
    return blob[:-1].split(b"\n")


class CaseRulesRef:
    """scan(text) -> (pos int64, ids int64) of the set of pattern file `blob` with these rules (n_parts = 1)."""

    def __init__(self, blob, rules, width=256, escapes=False):
        pats = patterns_of(blob, escapes)
        rules = [1 if r else 0 for r in rules]
        assert len(rules) == len(pats)
        self.lens = np.array([0] + [len(p) for p in pats], dtype=np.int64)
        self.subs = []   # (oracle, line ids of its sub-file, fold the text)
        for cls in (1, 0):
            ids = np.array([i + 1 for i, r in enumerate(rules) if r == cls], dtype=np.int64)
            if not len(ids):
                continue
            sub = [fold(pats[i - 1]) if cls else pats[i - 1] for i in ids]
            if escapes:
                o = Oracle(octal_file(sub), 1, width, escapes=True)
            else:
                o = Oracle(b"".join(p + b"\n" for p in sub), 1, width)
            self.subs.append((o, ids, cls == 1))

    def scan(self, text):
        text = np.ascontiguousarray(text, dtype=np.uint8)
        pos, ids = [np.zeros(0, np.int64)], [np.zeros(0, np.int64)]
        for o, line_ids, folded in self.subs:
            p, i = o.scan(fold(text) if folded else text)
            pos.append(np.asarray(p, dtype=np.int64))
            ids.append(line_ids[np.asarray(i, dtype=np.int64) - 1])
        pos, ids = np.concatenate(pos), np.concatenate(ids)
        order = np.lexsort((ids, self.lens[ids], pos))
        return pos[order], ids[order]


def brute_force(pats, rules, text):
    """The definition, window by window: every live line at every position (a line is shadowed by a later line of
    the same rule that equals it under that rule)."""
    live = []
    for i, (p, r) in enumerate(zip(pats, rules)):
        key = fold(p) if r else p
        if any((rules[j] and r and fold(pats[j]) == key) or (not rules[j] and not r and pats[j] == key)
               for j in range(i + 1, len(pats))):
            continue
        live.append((i + 1, key, r))
    t = bytes(np.ascontiguousarray(text, dtype=np.uint8))
    ft = fold(t)
    out = []
    for pos in range(len(t)):
        for i, key, r in live:
            src = ft if r else t
            if src[pos:pos + len(key)] == key:
                out.append((pos, len(key), i))
    out.sort()
    return (np.array([o[0] for o in out], dtype=np.int64), np.array([o[2] for o in out], dtype=np.int64))
