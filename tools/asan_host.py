#!/usr/bin/env python
"""Host code (table builder, derived filter tables, synthetic generators, writer) under
AddressSanitizer + UBSan.  No GPU, no CUDA: the four host translation units are built on their own.

    g++ -std=c++17 -O1 -g -fsanitize=address,undefined -fPIC -shared -Iinclude -Iphfpfac_b200/csrc -pthread \
        -o /tmp/libpfac_host_asan.so phfpfac_b200/csrc/pfac_{tables,writer,derive}.cc tools/synth/pfac_synth.cc
    LD_PRELOAD=$(gcc -print-file-name=libasan.so):$(gcc -print-file-name=libubsan.so) ASAN_OPTIONS=detect_leaks=0 \
        python tools/asan_host.py /tmp/libpfac_host_asan.so
Without an argument the tool builds that library and re-runs itself under the sanitizer runtimes.
Development tool; last run clean (round 2, final build)."""
import ctypes as C, sys, os, numpy as np, gzip, json, subprocess
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if len(sys.argv) < 2:
    so = "/tmp/libpfac_host_asan.so"
    src = [os.path.join(ROOT, "phfpfac_b200", "csrc", f"pfac_{n}.cc") for n in ("tables", "writer", "derive")] + [os.path.join(ROOT, "tools", "synth", "pfac_synth.cc")]
    subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-fPIC", "-shared",
                    "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "phfpfac_b200", "csrc"), "-I" + os.path.join(ROOT, "tools", "synth"),
                    "-pthread", "-o", so] + src, check=True)
    pre = ":".join(subprocess.run(["gcc", "-print-file-name=" + n], capture_output=True, text=True, check=True).stdout.strip() for n in ("libasan.so", "libubsan.so"))
    sys.exit(subprocess.run([sys.executable, os.path.abspath(__file__), so], env=dict(os.environ, LD_PRELOAD=pre, ASAN_OPTIONS="detect_leaks=0")).returncode)
lib = C.CDLL(sys.argv[1])
vp = C.c_void_p
lib.pfac_tables_build_mem_ext.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.c_int, C.c_uint, C.POINTER(vp)]
lib.pfac_tables_destroy.argtypes = [vp]
lib.pfac_tables_derive_check.argtypes = [vp, C.c_int, C.c_uint, C.c_uint, C.c_uint, C.POINTER(C.c_uint64)]
lib.pfac_last_error.restype = C.c_char_p
lib.pfac_synth_patterns.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_char_p, C.c_size_t]
lib.pfac_synth_patterns.restype = C.c_longlong
def synth(kind, n, seed, lo, hi):
    need = lib.pfac_synth_patterns(kind, n, seed, lo, hi, None, 0)
    buf = C.create_string_buffer(need)
    assert lib.pfac_synth_patterns(kind, n, seed, lo, hi, buf, need) == need
    return buf.raw[:need]
rng = np.random.default_rng(1)
cases = [(b"aaaa\naa\na\naaa\n", 0), (gzip.decompress(open(os.path.join(ROOT, 'tests', 'golden', 'dictionary.txt.gz'), 'rb').read()), 0),
         (synth(1, 3000, 3, 4, 64), 0), (synth(0, 20000, 5, 8, 32), 0), (b"a\\x41\\n\\\nb\\0c\n", 1), (b"abc\n\nabd\n", 0), (b"abc", 0), (b"", 0),
         (b"x" * 1023 + b"\n", 0), (b"\\", 1), (b"ab\\", 1)]
for t in range(30):
    n = int(rng.integers(1, 300)); lines = set()
    while len(lines) < n:
        L = int(rng.integers(1, 20)); lines.add(bytes((rng.integers(0, 255, L) + 0).astype(np.uint8)).replace(b"\n", b"\x0b"))
    cases.append((b"".join(l + b"\n" for l in lines), 0))
for blob, flags in cases:
    for width in (1, 8, 256, 4096):
        for parts in (1, 3):
            h = vp()
            rc = lib.pfac_tables_build_mem_ext(blob, len(blob), parts, width, flags, C.byref(h))
            if rc == 0:
                st = (C.c_uint64 * 10)()
                for sizes in ((32768, 32768, 32768), (1024, 0, 0), (131072, 4096, 256)):
                    rc2 = lib.pfac_tables_derive_check(h, 0, *sizes, st)
                    assert rc2 == 0, (rc2, lib.pfac_last_error())
                lib.pfac_tables_destroy(h)
print("asan drive ok", len(cases))
# writer + synth text
lib.pfac_synth_text.argtypes = [C.c_int, C.c_uint64, C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int]
pats = synth(1, 500, 3, 4, 64)
for n in (0, 1, 65535, 65536, 300001):
    buf = np.zeros(max(n, 1), dtype=np.uint8)
    assert lib.pfac_synth_text(1, 7, buf.ctypes.data, n, pats, len(pats), 3) == 0
    assert lib.pfac_synth_text(0, 7, buf.ctypes.data, n, None, 0, 0) == 0
lib.pfac_format_records.restype = C.c_size_t
lib.pfac_format_records.argtypes = [C.c_uint64, C.c_void_p, C.c_uint64, C.c_char_p, C.c_size_t]
rec = np.zeros((1 << 20) + 77, dtype=[("pos", "<u4"), ("id", "<u4")]); rec["pos"] = np.arange(len(rec)) * 5; rec["id"] = np.arange(len(rec)) % 1000 + 1
for base in (0, 2 ** 40 + 3):
    need = lib.pfac_format_records(base, rec.ctypes.data, len(rec), None, 0)
    out = C.create_string_buffer(need)
    assert lib.pfac_format_records(base, rec.ctypes.data, len(rec), out, need) == need
lib.pfac_write_begin.argtypes = [C.c_char_p, C.POINTER(vp)]; lib.pfac_write_records.argtypes = [vp, C.c_uint64, C.c_void_p, C.c_uint64]; lib.pfac_write_end.argtypes = [vp]
w = vp(); assert lib.pfac_write_begin(b"/tmp/asan_out.txt", C.byref(w)) == 0
assert lib.pfac_write_records(w, 9, rec.ctypes.data, len(rec)) == 0 and lib.pfac_write_records(w, 9, rec.ctypes.data, 10) == 0
assert lib.pfac_write_end(w) == 0
print("asan writer/synth ok")
# binary sidecar: write, read back, damaged files
lib.pfac_sidecar_begin.argtypes = [C.c_char_p, C.POINTER(vp)]; lib.pfac_sidecar_records.argtypes = [vp, C.c_uint64, C.c_void_p, C.c_uint64]; lib.pfac_sidecar_end.argtypes = [vp]
lib.pfac_sidecar_read.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
sc = vp(); assert lib.pfac_sidecar_begin(b"/tmp/asan_side.bin", C.byref(sc)) == 0
assert lib.pfac_sidecar_records(sc, 2 ** 40, rec.ctypes.data, len(rec)) == 0 and lib.pfac_sidecar_records(sc, 2 ** 41, rec.ctypes.data, 10) == 0 and lib.pfac_sidecar_records(sc, 0, None, 0) == 0
assert lib.pfac_sidecar_end(sc) == 0
n = C.c_uint64(0); assert lib.pfac_sidecar_read(b"/tmp/asan_side.bin", None, None, 0, C.byref(n)) == 0 and n.value == len(rec) + 10
pos = np.zeros(n.value, dtype=np.uint64); ids = np.zeros(n.value, dtype=np.uint32)
assert lib.pfac_sidecar_read(b"/tmp/asan_side.bin", pos.ctypes.data, ids.ctypes.data, n.value, C.byref(n)) == 0
assert pos[0] == 2 ** 40 and pos[-1] == 2 ** 41 + 45 and ids[-1] == 10
assert lib.pfac_sidecar_read(b"/tmp/asan_side.bin", pos.ctypes.data, None, n.value - 1, C.byref(n)) == -8
raw = open("/tmp/asan_side.bin", "rb").read()
for cut in (0, 7, 31, 32, 40, 48, 49, len(raw) - 1):
    open("/tmp/asan_side_bad.bin", "wb").write(raw[:cut])
    assert lib.pfac_sidecar_read(b"/tmp/asan_side_bad.bin", pos.ctypes.data, ids.ctypes.data, n.value, C.byref(n)) == -1, cut
for off in (16, 24, 40):   # block count / record count / a block's count: every inconsistency is an I/O error, never an overrun
    bad = bytearray(raw); bad[off:off + 8] = (2 ** 50).to_bytes(8, "little")
    open("/tmp/asan_side_bad.bin", "wb").write(bytes(bad))
    rc = lib.pfac_sidecar_read(b"/tmp/asan_side_bad.bin", pos.ctypes.data, ids.ctypes.data, len(pos), C.byref(n))
    assert rc in (-1, -8), (off, rc)
print("asan sidecar ok")
# table cache: save / load round trip and damaged files
lib.pfac_tables_save.argtypes = [vp, C.c_char_p]; lib.pfac_tables_load.argtypes = [C.c_char_p, C.POINTER(vp)]
blob = synth(1, 2000, 9, 4, 48)
h = vp(); assert lib.pfac_tables_build_mem_ext(blob, len(blob), 2, 256, 0, C.byref(h)) == 0
assert lib.pfac_tables_save(h, b"/tmp/asan_tables.bin") == 0
h2 = vp(); assert lib.pfac_tables_load(b"/tmp/asan_tables.bin", C.byref(h2)) == 0
lib.pfac_tables_destroy(h2)
raw = open("/tmp/asan_tables.bin", "rb").read()
for t in range(200):
    bad = bytearray(raw)
    if t % 2:
        bad = bad[:int(rng.integers(0, len(bad)))]
    else:
        for k in range(int(rng.integers(1, 4))):
            bad[int(rng.integers(0, len(bad)))] ^= 1 << int(rng.integers(0, 8))
    open("/tmp/asan_tables_bad.bin", "wb").write(bytes(bad))
    h2 = vp()
    if lib.pfac_tables_load(b"/tmp/asan_tables_bad.bin", C.byref(h2)) == 0:
        lib.pfac_tables_destroy(h2)   # (a flipped bit in unused padding may load)
lib.pfac_tables_destroy(h)
print("asan table cache ok")
# per-pattern case rules: mixed builds (escapes included), lengths, save / load and damaged files
lib.pfac_tables_build_mem_rules.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.c_int, C.c_uint, C.c_void_p, C.c_uint32, C.POINTER(vp)]
lib.pfac_tables_pattern_lengths.argtypes = [vp, C.c_int, C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]
lib.pfac_tables_case_rules.argtypes = [vp, C.c_void_p, C.c_uint32]
lib.pfac_tables_n_patterns.argtypes = [vp]
mixed = [(b"GET\nget\nGeT\nGET\n123\nget\n", 0), (b"a\\x41\\n\\\nb\\0c\nA\\x61\n", 1), (synth(1, 3000, 3, 4, 64), 0),
         (b"x" * 1022 + b"\n" + b"X" * 1022 + b"\n", 0), (b"ab\nAB\n", 1), (b"", 0), (b"abc", 0)]
for blob, flags in mixed:
    n_pat = blob.count(b"\n") if not flags else 2
    for parts in (1, 3):
        rules = (np.arange(max(n_pat, 1)) % 3 == 0).astype(np.uint8)
        h = vp()
        rc = lib.pfac_tables_build_mem_rules(blob, len(blob), parts, 256, flags, rules.ctypes.data, n_pat, C.byref(h))
        if rc != 0:
            continue
        got = np.zeros(lib.pfac_tables_n_patterns(h), dtype=np.uint8)
        assert lib.pfac_tables_case_rules(h, got.ctypes.data, len(got)) == 0
        for g in range(parts):
            nid = C.c_int32(0)
            assert lib.pfac_tables_pattern_lengths(h, g, None, 0, C.byref(nid)) == 0
            lens = np.zeros(max(nid.value, 1), dtype=np.int32)
            assert lib.pfac_tables_pattern_lengths(h, g, lens.ctypes.data, len(lens), C.byref(nid)) == 0
        assert lib.pfac_tables_save(h, b"/tmp/asan_rules.bin") == 0
        h2 = vp(); assert lib.pfac_tables_load(b"/tmp/asan_rules.bin", C.byref(h2)) == 0
        lib.pfac_tables_destroy(h2)
        raw = open("/tmp/asan_rules.bin", "rb").read()
        for t in range(60):
            bad = bytearray(raw)
            if t % 2:
                bad = bad[:int(rng.integers(0, len(bad)))]
            else:
                bad[int(rng.integers(0, len(bad)))] ^= 1 << int(rng.integers(0, 8))
            open("/tmp/asan_rules_bad.bin", "wb").write(bytes(bad))
            h2 = vp()
            if lib.pfac_tables_load(b"/tmp/asan_rules_bad.bin", C.byref(h2)) == 0:
                lib.pfac_tables_destroy(h2)
        lib.pfac_tables_destroy(h)
print("asan case rules ok")
