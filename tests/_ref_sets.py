"""The seeded inputs of the comparisons with the reference itself, shared by the tests and by
tests/golden/make_ref_live.py, which stores what the reference computed on them in tests/golden/ref_live.json."""
import numpy as np

import pfac_synth as synth
from bench import WORKLOADS


def random_patterns(rng, n, alpha, max_len, base=97):
    pats = set()
    while len(pats) < n:
        L = int(rng.integers(1, max_len + 1))
        pats.add(bytes((rng.integers(0, alpha, L) + base).astype(np.uint8)))
    pats = sorted(pats)      # a set's order changes from process to process (hash randomisation)
    rng.shuffle(pats)
    return b"".join(p + b"\n" for p in pats)


def oracle_builder_sets():
    """-> [(pattern file image, streamnum, width)]: random sets through create_PFAC_table_reorder + FFDM
    (streamnum 1 or 2: 4 or 8 partitions), widths 1..4096."""
    rng = np.random.default_rng(7)
    out = []
    for trial in range(6):
        n = int(rng.integers(5, 400))
        alpha = int(rng.integers(2, 40))
        pats = set()
        while len(pats) < n:
            L = int(rng.integers(1, 12))
            pats.add(bytes((rng.integers(0, alpha, L) + 97).astype(np.uint8)))
        blob = b"".join(p + b"\n" for p in sorted(sorted(pats), key=lambda _: rng.random()))
        width = int(2 ** rng.integers(0, 13))
        out.append((blob, 1 + trial % 2, width))
    return out


def product_builder_sets():
    """-> [(pattern file image, width)]: built in 4 partitions (streamnum 1) and as one automaton."""
    rng = np.random.default_rng(17)
    out = []
    for _ in range(4):
        blob = random_patterns(rng, int(rng.integers(10, 600)), int(rng.integers(2, 60)), 14)
        out.append((blob, int(2 ** rng.integers(3, 13))))
    return out


def gpu_kernel_case(mib=3):
    """-> (patterns, text): bench.py's config-3 pattern set over the first `mib` MiB of its text, the input of
    tests/refgpu_bench.py --mib 3 (the reference's dense result indexes at most 16 MiB of it)."""
    pk, cnt, pseed, lo, hi, tk, tseed, _n, _d = WORKLOADS["config3"]
    pats = synth.synth_patterns(pk, cnt, pseed, lo, hi)
    return pats, synth.synth_text(tk, tseed, mib << 20, patterns=pats)
