"""Reference for caseless pattern sets (PFAC_PATTERNS_CASELESS, this project's flag: the reference has no
case-insensitive mode), built on the unchanged oracle (tests/_oracle.py).

A caseless set is the set of its patterns, as the reader returns them, folded ('A'-'Z' -> 'a'-'z', no other byte)
before the sort.  Without escapes that is the oracle's build of the folded file.  With PFAC_PATTERNS_ESCAPES the file
cannot simply be folded (an escaped \\x41 would still read as 'A'), so the patterns are decoded here -- a Python
restatement of the escape reader (ctdef.h:37-99 fgetc_ext, create_table_reorder.c:131-185 read_pattern_ext) -- then
folded, and handed back to the oracle's escape reader with every byte written as a three-digit octal escape, in file
order (so ids and the last-duplicate-wins rule are the oracle's own)."""
import numpy as np

from _oracle import Oracle

FOLD = bytes(b + 0x20 if 0x41 <= b <= 0x5A else b for b in range(256))
FOLD_NP = np.frombuffer(FOLD, dtype=np.uint8)


def fold(data):
    """The fold of bytes (-> bytes) or of a uint8 array (-> a new array)."""
    if isinstance(data, np.ndarray):
        return FOLD_NP[data]
    return bytes(data).translate(FOLD)


_ESC = {ord("a"): 7, ord("b"): 8, ord("t"): 9, ord("n"): 10, ord("v"): 11, ord("f"): 12, ord("r"): 13,
        ord("'"): 39, ord('"'): 34, ord("\\"): 92}
_EOL = -2


def _next(buf, i):
    """fgetc_ext over a buffer: (byte or _EOL, next index).  \\ooo: up to 3 octal digits; \\xhh: white space skipped,
    up to 2 hex digits; the named escapes; any other backslash stays a backslash (the next byte is read again)."""
    c0 = buf[i]
    i += 1
    if c0 == 0x5C and i < len(buf):
        c1 = buf[i]
        if 0x30 <= c1 <= 0x39:
            v = nd = 0
            while nd < 3 and i < len(buf) and 0x30 <= buf[i] <= 0x37:
                v, i, nd = v * 8 + buf[i] - 0x30, i + 1, nd + 1
            return v & 255, i
        if c1 in _ESC:
            return _ESC[c1], i + 1
        if c1 == ord("x"):
            i += 1
            while i < len(buf) and (buf[i] == 0x20 or 9 <= buf[i] <= 13):
                i += 1
            v = nd = 0
            while nd < 2 and i < len(buf) and chr(buf[i]) in "0123456789abcdefABCDEF":
                v, i, nd = v * 16 + int(chr(buf[i]), 16), i + 1, nd + 1
            return v & 255, i
        return c0, i
    return (_EOL if c0 == 10 else c0), i


def decode_escapes(blob):
    """The patterns of a well-formed escaped pattern file (every line ends with a raw newline), in file order."""
    pats, cur, i = [], bytearray(), 0
    while i < len(blob):
        c, i = _next(blob, i)
        if c == _EOL:
            pats.append(bytes(cur))
            cur = bytearray()
        else:
            cur.append(c)
    assert not cur, "pattern file must end with a newline"
    return pats


def octal_file(pats):
    """An escaped pattern file that the escape reader reads back as exactly these patterns, in this order."""
    return b"".join(b"".join(b"\\%03o" % c for c in p) + b"\n" for p in pats)


def caseless_oracle(blob, n_parts=4, width=256, escapes=False):
    """The oracle of the caseless set of pattern file `blob`."""
    if not escapes:
        return Oracle(fold(blob), n_parts, width)
    return Oracle(octal_file([fold(p) for p in decode_escapes(blob)]), n_parts, width, escapes=True)
