"""CPU: the C-ABI boundary — the shared objects load, export exactly what include/b200bgzf.h declares (and
nothing unprefixed besides bgzf_compress), and fail loudly without a GPU (no CPU fallback)."""
import ctypes
import glob
import json
import os
import re
import subprocess
import sys

import pytest

import b200bgzf
import helpers as H

ROOT = H.ROOT
HAVE_GPU = bool(glob.glob("/dev/nvidia[0-9]*"))        # a machine may expose its GPU under any index, not only 0


def _declared():
    hdr = open(os.path.join(ROOT, "include", "b200bgzf.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(b200bgzf_\w+|bgzf_compress)\s*\(", hdr)))


def _exported(path):
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    return sorted(l.split()[-1] for l in out.splitlines() if " T " in l)


def test_built():
    for p in (b200bgzf.LIB_PATH, b200bgzf.HOOK_PATH, b200bgzf.APPLET_PATH):
        assert os.path.exists(p), f"{p} missing: run make"


def test_library_exports_match_header():
    decl = _declared()
    assert "bgzf_compress" in decl and len(decl) >= 14
    assert _exported(b200bgzf.HOOK_PATH) == decl                       # 7bgzf.so: the hook + the prefixed API, nothing else
    assert _exported(b200bgzf.LIB_PATH) == [d for d in decl if d != "bgzf_compress"]
    lib = b200bgzf.load()
    for name in b200bgzf.EXPORTS:
        assert hasattr(lib, name)


def test_no_foreign_symbols_interposed():
    # the reference .so exports 600+ symbols (deflate, inflate, crc32, main, finish ...); ours must not
    names = _exported(b200bgzf.HOOK_PATH)
    for bad in ("deflate", "inflate", "crc32", "main", "finish", "libdeflate_deflate_compress"):
        assert bad not in names


def test_parse_method_matches_reference_levels():
    lib = b200bgzf.load()
    lvl, olvl = ctypes.c_int(), ctypes.c_int()
    name = ctypes.create_string_buffer(32)
    for spec in (None, b"", b"libdeflate", b"LIBDEFLATE12", b"libdeflate1", b"zlib", b"zlib9", b"slz", b"7-zip", b"igzip3", b"bogus7", b"zopfli", b"miniz2"):
        assert lib.b200bgzf_parse_method(spec, ctypes.byref(lvl), name, 32) == 0
        H.oracle().oracle_parse_method(spec, ctypes.byref(olvl))
        assert lvl.value == max(1, olvl.value), spec          # same level the reference's parser yields
    assert lib.b200bgzf_parse_method(b"libdeflate13", ctypes.byref(lvl), name, 32) == -1   # reference: NULL deref
    assert lib.b200bgzf_parse_method(b"libdeflate", ctypes.byref(lvl), name, 32) == 0 and name.value == b"libdeflate"


def test_bound_and_errors():
    lib = b200bgzf.load()
    assert lib.b200bgzf_compress_bound(0, 0xFF00) == 28
    assert lib.b200bgzf_compress_bound(65280, 0xFF00) >= 65311 + 28
    assert lib.b200bgzf_compress_bound(10, 0x10001) == 0
    assert b"fit" in lib.b200bgzf_strerror(1)


def test_hook_paths_that_need_no_gpu():
    hook = ctypes.CDLL(b200bgzf.HOOK_PATH)
    hook.bgzf_compress.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_size_t), ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int]
    dst = ctypes.create_string_buffer(64)
    n = ctypes.c_size_t(64)
    assert hook.bgzf_compress(dst, ctypes.byref(n), b"", 0, 6) == 0 and n.value == 28 and dst.raw[:28] == H.EOF_BLOCK
    n = ctypes.c_size_t(27)
    assert hook.bgzf_compress(dst, ctypes.byref(n), b"", 0, 6) == -1 and n.value == 27


@pytest.mark.skipif(HAVE_GPU, reason="this checks the no-GPU behaviour")
def test_no_cpu_fallback_without_gpu():
    with pytest.raises(b200bgzf.B200BgzfError):
        b200bgzf.Codec()
    r = subprocess.run([b200bgzf.APPLET_PATH, "-c", "-l6"], input=b"hello", capture_output=True)
    assert r.returncode != 0 and r.stdout == b"" and b"cannot initialise the GPU codec" in r.stderr
    # the hook must not quietly compress on the CPU either
    code = ("import ctypes,sys; h=ctypes.CDLL(sys.argv[1]); d=ctypes.create_string_buffer(65536); n=ctypes.c_size_t(65536);"
            "h.bgzf_compress.argtypes=[ctypes.c_char_p,ctypes.POINTER(ctypes.c_size_t),ctypes.c_char_p,ctypes.c_size_t,ctypes.c_int];"
            "print(h.bgzf_compress(d,ctypes.byref(n),b'x'*1000,1000,6), n.value)")
    r = subprocess.run([sys.executable, "-c", code, b200bgzf.HOOK_PATH], capture_output=True, text=True, env=dict(os.environ, BGZF_METHOD="libdeflate6"))
    assert r.stdout.split() == ["-1", "65536"]


def test_applet_cli_contract():
    r = subprocess.run([b200bgzf.APPLET_PATH], input=b"", capture_output=True)
    assert r.returncode == 1 and b"Usage" in r.stderr                    # no method, no -d  (7bgzf.c:467-479)
    r = subprocess.run([b200bgzf.APPLET_PATH, "-l6", "-z"], input=b"", capture_output=True)
    assert r.returncode == 1                                             # two methods
    r = subprocess.run([b200bgzf.APPLET_PATH, "-d", "-l6"], input=b"", capture_output=True)
    assert r.returncode == 1                                             # method together with -d


def test_thread_pool_harness_against_the_reference_hook(tmp_path):
    """build/hook_mt (the stand-in for htslib's pool used for the hook numbers) drives any .so that exports
    bgzf_compress: here the reference's, on CPU; and it fails cleanly on the GPU hook when there is no GPU."""
    exe = os.path.join(H.ROOT, "build", "hook_mt")
    if not os.path.exists(exe) or not H.have_ref():
        pytest.skip("build/hook_mt or oracle/_ref missing")
    f = tmp_path / "in.sam"
    f.write_bytes(H.synth("sam", 6 * H.BLOCK + 123))
    env = dict(os.environ, BGZF_METHOD="libdeflate6")
    r = subprocess.run([exe, H.REF_SO, "3", str(f)], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    out = json.loads(r.stdout)
    assert out["threads"] == 3 and out["bytes"] == 6 * H.BLOCK + 123 and 0.05 < out["ratio"] < 0.3
    r = subprocess.run([exe, b200bgzf.HOOK_PATH, "2", str(f)], capture_output=True, text=True, env=env)
    try:
        b200bgzf.Codec().close()
        assert r.returncode == 0, r.stderr                           # (a GPU is present: the hook works)
    except b200bgzf.B200BgzfError:
        assert r.returncode != 0 and "failed" in r.stderr        # no GPU here: every call returns -1, nothing is faked


def _gz_member(payload, flavour, level=6, name=None):
    """one gzip member in a block-gzip flavour the reference's decompress loop accepts (applet/7bgzf.c:81-131)"""
    import struct, zlib
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    raw = co.compress(payload) + co.flush()
    tail = struct.pack("<II", zlib.crc32(payload), len(payload) & 0xffffffff)
    flags = 4 | (8 if name else 0)
    fixed = bytes([0x1f, 0x8b, 8, flags, 0, 0, 0, 0, 0, 0xff])
    nm = (name + b"\0") if name else b""
    def build(extra):
        return fixed + struct.pack("<H", len(extra)) + extra + nm + raw + tail
    if flavour == "bgzf":
        total = len(build(b"BC\x02\x00\0\0"))
        return build(b"BC\x02\x00" + struct.pack("<H", total - 1))
    if flavour == "migz":
        return build(b"MZ\x04\x00" + struct.pack("<I", len(raw)))
    if flavour == "mgzip2":
        total = len(build(b"IG\x04\x00\0\0\0\0"))
        return build(b"IG\x04\x00" + struct.pack("<I", total))
    if flavour == "mgzip1":
        total = len(build(b"IG\x10\x00" + bytes(16)))
        return build(b"IG\x10\x00" + struct.pack("<QQ", total, len(payload)))
    raise ValueError(flavour)


def test_member_header_parser_matches_the_oracle_and_the_reference_decoder(tmp_path):
    """b200bgzf_member_header (product) against oracle_read_gz_header (restatement of applet/7bgzf.c:81-131) on every
    flavour, with and without a name field, on truncations and on mutated bytes; and the reference applet itself
    decodes the fixtures this test builds, so the fixtures are what the reference means by these formats."""
    import random
    lib = b200bgzf.load()
    o = H.oracle()
    payload = H.synth("sam", 70000)
    eo, el, bl = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    rnd = random.Random(7)
    for flavour in ("bgzf", "migz", "mgzip1", "mgzip2"):
        for name in (None, b"file.txt"):
            m = _gz_member(payload[:40000] if flavour == "bgzf" else payload, flavour, name=name)
            want = o.oracle_read_gz_header(m, len(m), eo, el, bl)
            assert want > 0 and bl.value == len(m), (flavour, name)
            assert b200bgzf.member_header(m, lib) == (want, len(m))
            assert b200bgzf.member_header(m + b"trailing", lib) == (want, len(m))
            assert b200bgzf.member_header(m[:-1], lib) == (0, 0)                    # cut short: not a whole member
            for _ in range(200):                                                     # mutated headers: same verdict as the oracle
                bad = bytearray(m)
                k = rnd.randrange(0, want)
                bad[k] ^= 1 << rnd.randrange(8)
                bad = bytes(bad)
                w = o.oracle_read_gz_header(bad, len(bad), eo, el, bl)
                got = b200bgzf.member_header(bad, lib)
                if w > 0 and want + 8 <= bl.value <= len(bad):
                    assert got == (w, bl.value), (flavour, k)
                else:
                    assert got == (0, 0), (flavour, k)
    assert b200bgzf.member_header(b"\x1f\x8b\x08\x00" + bytes(40), lib) == (0, 0)       # plain gzip: no block length
    if H.have_ref():
        stream = b"".join(_gz_member(payload, f) for f in ("migz", "mgzip2", "mgzip1")) + _gz_member(payload[:30000], "bgzf")
        r = subprocess.run([os.path.join(H.ROOT, "oracle", "_ref", "7bgzf"), "-d"], input=stream, capture_output=True)
        assert r.returncode == 0 and r.stdout == payload * 3 + payload[:30000]


def test_gzi_formatter_layout():
    """b200bgzf_gzi_format: u64 count then (caddr, uaddr) of every member but the first, little endian (htslib .gzi)"""
    import struct
    assert b200bgzf.gzi_format([], []) == struct.pack("<Q", 0)
    assert b200bgzf.gzi_format([0], [0]) == struct.pack("<Q", 0)
    ca, ua = [0, 1234, 70000, 2**33 + 5], [0, 65280, 130560, 2**34 + 7]
    want = struct.pack("<Q", 3) + b"".join(struct.pack("<QQ", c, u) for c, u in zip(ca[1:], ua[1:]))
    assert b200bgzf.gzi_format(ca, ua) == want
    # too small a destination writes nothing
    lib = b200bgzf.load()
    import ctypes
    a = (ctypes.c_uint64 * 4)(*ca)
    b = (ctypes.c_uint64 * 4)(*ua)
    buf = bytearray(8 + 16 * 3 - 1)
    assert lib.b200bgzf_gzi_format(a, b, 4, b200bgzf._addr(buf), len(buf)) == 0
    # and the header-walk oracle of tests/helpers.py agrees on a hand-made stream (zlib-made members)
    stream = b"".join(H.zlib_member(pl) for pl in (b"a" * 100, b"b" * 7, b"c" * 5000)) + b200bgzf.EOF_BLOCK
    offs = [m[0] for m in H.members(stream)][:3]
    assert H.gzi_of(stream) == b200bgzf.gzi_format(offs, [0, 100, 107])


def test_shard_blocks_partition_is_contiguous_and_complete():
    """b200bgzf_shard_blocks (the rule of SURVEY 8e: GPU g of G takes blocks [B*g/G, B*(g+1)/G)) == shard.block_range"""
    import shard
    for nb in (0, 1, 7, 16449, 1052689, (1 << 40) + 12345):
        for world in (1, 2, 3, 4, 8, 64):
            cuts = [b200bgzf.shard_blocks(nb, r, world) for r in range(world)]
            assert cuts[0][0] == 0 and cuts[-1][1] == nb
            assert all(cuts[r][1] == cuts[r + 1][0] for r in range(world - 1))
            assert cuts == [shard.block_range(nb, r, world) for r in range(world)]


def test_multi_create_without_gpu_fails_loudly():
    if HAVE_GPU:
        pytest.skip("GPU present")
    with pytest.raises(b200bgzf.B200BgzfError) as e:
        b200bgzf.MultiCodec([0, 1])
    assert e.value.code == b200bgzf.E_CUDA
