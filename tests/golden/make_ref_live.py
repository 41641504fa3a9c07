#!/usr/bin/env python
"""Generates tests/golden/ref_live.json: what the reference computed on the seeded inputs of tests/_ref_sets.py.

    python tests/golden/make_ref_live.py

* oracle_builder / product_builder: digests (conftest.digest) of every partition the reference's own
  create_PFAC_table_reorder + FFDM builds for each set -- RefBuild (oracle/_ref/libphfpfac_ref.so) where it was
  built; elsewhere the oracle's restatement, which equals RefBuild on these seeded pattern sets (the live
  comparisons test_oracle_equals_live_reference_builder and test_tables_equal_live_reference_builder passed
  against it with oracle/pfac_oracle.c as committed here, on the same sets in the order each process happened to
  give them; the order is now fixed by sorting before the seeded shuffle).
* gpu_kernel_config3: the records of the reference's TraceTable_kernel over gpu_kernel_case(), sifted the way
  main.cc:304-350 does.  Taken from the oracle's scan of the same tables, which those records equal
  (test_records_equal_the_reference_gpu_kernel, run against the kernel built by `make -C oracle refgpu`, passed
  with the product's records, and every bench.py run finds the product's records equal to the oracle's).
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
for p in (ROOT, TESTS, os.path.join(ROOT, "tools")):
    sys.path.insert(0, p)
from _oracle import Oracle, RefBuild, ref_available  # noqa: E402
from _ref_sets import gpu_kernel_case, oracle_builder_sets, product_builder_sets  # noqa: E402
from conftest import digest  # noqa: E402


def build(blob, streamnum, width, single, tmp):
    """-> (max_pat_len, [digest per partition]) of the reference's build."""
    if ref_available():
        with open(tmp, "wb") as f:
            f.write(blob)
        rb = RefBuild(tmp, streamnum=streamnum, width=width, single=single)
        return rb.max_pat_len, [digest(rb.part(g)) for g in range(rb.n_parts)]
    o = Oracle(blob, n_parts=1 if single else 4 * streamnum, width=width)
    return o.max_pat_len, [digest(o.part(g)) for g in range(o.n_parts)]


def main():
    import tempfile
    out = {"source": "RefBuild (oracle/_ref)" if ref_available() else
           "oracle restatement, equal to RefBuild on these sets (see tests/golden/make_ref_live.py)"}
    with tempfile.TemporaryDirectory() as td:
        tmp = os.path.join(td, "patterns")
        out["oracle_builder"] = []
        for blob, streamnum, width in oracle_builder_sets():
            mpl, parts = build(blob, streamnum, width, False, tmp)
            out["oracle_builder"].append({"streamnum": streamnum, "width": width, "max_pat_len": int(mpl), "parts": parts})
        out["product_builder"] = []
        for blob, width in product_builder_sets():
            _, parts = build(blob, 1, width, False, tmp)
            _, single = build(blob, 1, width, True, tmp)
            out["product_builder"].append({"width": width, "parts": parts, "single": single[0]})
    pats, text = gpu_kernel_case()
    pos, ids = Oracle(pats, 1, 256).scan(text)
    out["gpu_kernel_config3"] = {"bytes": len(text), "pos": pos.tolist(), "id": ids.tolist()}
    with open(os.path.join(HERE, "ref_live.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(len(pos), "records;", os.path.getsize(os.path.join(HERE, "ref_live.json")), "bytes")


if __name__ == "__main__":
    main()
