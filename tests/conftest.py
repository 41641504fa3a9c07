"""Shared fixtures.  `-m "not gpu"`: oracle vs goldens, host logic, ABI surface (no compute calls).
`-m gpu`: parity of the CUDA path (through the C ABI) with the oracle."""
import gzip
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
for p in (ROOT, HERE, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run by the driver on the GPU box)")
    # the product library and the checkers are built artefacts (git-ignored): build them once
    lib = os.path.join(ROOT, "phfpfac_b200", "_build", "libpfac_b200.so")
    if not os.path.exists(lib):
        subprocess.run(["make", "-s", "-C", ROOT, "lib", "cli"], check=True)
    if not os.path.exists(os.path.join(ROOT, "tools", "_build", "libpfac_synth.so")):
        subprocess.run(["make", "-s", "-C", ROOT, "synth"], check=True)
    if not os.path.exists(os.path.join(ROOT, "oracle", "_build", "libpfac_oracle.so")):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "oracle"], check=True)


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no GPU in this container (runs under gpurun / the driver's GPU tier)")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_fixtures():
    fx = json.load(open(os.path.join(GOLDEN, "fixtures.json")))
    out = {
        "experimentpattern": bytes.fromhex(fx["experimentpattern_hex"]),
        "experimentinput": bytes.fromhex(fx["experimentinput_hex"]),
    }
    period = bytes.fromhex(fx["one_m_period_hex"])
    one_m = (period * (fx["one_m_size"] // len(period) + 1))[:fx["one_m_size"]]
    assert hashlib.sha256(one_m).hexdigest() == fx["one_m_sha256"]
    out["1M"] = one_m
    d = gzip.decompress(open(os.path.join(GOLDEN, "dictionary.txt.gz"), "rb").read())
    assert hashlib.sha256(d).hexdigest() == fx["dictionary_sha256"]
    out["dictionary"] = d
    off = 0
    for name in ("xaa", "xab", "xac", "xad"):
        n = fx["dictionary_parts"][name]
        out[name] = d[off:off + n]
        off += n
    return out


@pytest.fixture(scope="session")
def fixtures():
    return load_fixtures()


@pytest.fixture(scope="session")
def golden():
    return json.load(open(os.path.join(GOLDEN, "golden.json")))


@pytest.fixture(scope="session")
def ref_live():
    """What the reference computed on the seeded inputs of _ref_sets.py (tests/golden/make_ref_live.py)."""
    return json.load(open(os.path.join(GOLDEN, "ref_live.json")))


def sha_i32(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.int32).tobytes()).hexdigest()


def digest(p):
    """Same digest as tests/golden/make_golden.py:table_digest."""
    return {"state_num": int(p.state_num), "n_final": int(p.n_final), "max_len": int(p.max_len),
            "ht_size": int(p.ht_size), "n_r": int(len(p.r)), "s0": sha_i32(p.s0), "r": sha_i32(p.r),
            "HT": sha_i32(p.HT), "val": sha_i32(p.val), "idmap": sha_i32(p.idmap)}


def parse_key(key):
    name, parts, width = key.split("|")
    return name, int(parts.split("=")[1]), int(width.split("=")[1])
