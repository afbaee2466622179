"""Whole-stream gzip members without usable flush points (GNU gzip, zlib's default deflate(), Python's gzip module), decoded
in parallel from DEFLATE block starts found by a search at bit offsets (DESIGN §6g): b200bgzf_container_inflate_host(GZIP) and
b200bgzf_gzip_inflate_device.  Every stream is checked against zlib and, where one warp finishes in seconds, against the
one-warp path, whose bytes or error code the searched route must reproduce exactly."""
import ctypes
import gzip
import io
import os
import random
import shutil
import struct
import subprocess
import sys
import zlib

import pytest

import b200bgzf as B
import helpers as H
from test_gzip_parallel import GZIP_EXE, device, one_warp, outcome, parallel, sync_flush_stream, with_header

gpu = pytest.mark.gpu
REGION = 256 << 10           # compressed bytes per search region
ROUNDS = 8                   # chain repairs before the member goes to one warp
CHAIN_LAUNCHES = 16          # a flush-point member in one batch: count 3, chain 8, batch 5


def zlib_member(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, mem=8, wbits=15):
    z = zlib.compressobj(level, zlib.DEFLATED, wbits + 16, mem, strategy)
    return z.compress(data) + z.flush()


def gnu_gzip(data, level):
    return subprocess.run(["gzip", "-c", "-n", "-%d" % level], input=data, capture_output=True, check=True).stdout


def python_gzip(data):
    buf = io.BytesIO()
    with gzip.GzipFile(filename="reads.fq", fileobj=buf, mode="wb", compresslevel=6, mtime=0) as f:
        f.write(data)
    return buf.getvalue()


def stored_stream(payload, sizes):
    """raw DEFLATE of stored blocks only, cutting payload into blocks of the given payload sizes (the last one final)"""
    out, at = [], 0
    for i, n in enumerate(sizes):
        final = i == len(sizes) - 1
        out.append(bytes([1 if final else 0]) + struct.pack("<HH", n, n ^ 0xFFFF) + payload[at : at + n])
        at += n
    assert at == len(payload)
    return b"".join(out)


def fill_sizes(nbytes):
    """stored-block payload sizes whose blocks (5 header bytes each) fill nbytes of DEFLATE data exactly"""
    blocks = [65540] * (nbytes // 65540)
    rest = nbytes % 65540
    if 0 < rest < 6:
        blocks[-1] -= 6
        rest += 6
    if rest:
        blocks.append(rest)
    return [n - 5 for n in blocks]


def region_sizes(nreg):
    """stored-block payload sizes for nreg regions, a block header at every region start"""
    return fill_sizes(REGION) * nreg


def mixed(mib, seed=1):
    """FASTQ- and SAM-like text, a noise stretch (stored blocks in the middle of the member) and zeros (high expansion)"""
    q = mib << 20
    return (H.synth("fastq", q * 3 // 8, seed=seed) + H.lcg_noise(200000) + H.synth("sam", q * 3 // 8, seed=seed + 1) +
            bytes(q // 4))


def launches(codec, blob, flags=0):
    before = codec.launches()
    device(codec, blob, flags)
    return codec.launches() - before


def one_warp_launches(codec):
    """what a member without flush points within one region costs: the flush-point count, then one warp"""
    return launches(codec, zlib_member(H.synth("fastq", 200000)))


def check(codec, blob, data, reference=True):
    assert zlib.decompress(blob, 31) == data
    for flags in (0, B.VERIFY):
        assert parallel(codec, blob, flags) == data
        assert device(codec, blob, flags) == data
    if reference:
        assert one_warp(codec, blob) == data


@pytest.fixture(scope="module")
def codec():
    c = B.Codec(0)
    yield c
    c.close()


# ---------------------------------------------------------------- 1. encoders


ENCODERS = [
    (1, zlib.Z_DEFAULT_STRATEGY, 8, 15),
    (6, zlib.Z_DEFAULT_STRATEGY, 8, 15),
    (9, zlib.Z_DEFAULT_STRATEGY, 8, 15),
    (6, zlib.Z_FILTERED, 8, 15),
    (6, zlib.Z_HUFFMAN_ONLY, 8, 15),
    (1, zlib.Z_RLE, 8, 15),
    (6, zlib.Z_DEFAULT_STRATEGY, 1, 15),
    (9, zlib.Z_DEFAULT_STRATEGY, 9, 15),
    (6, zlib.Z_DEFAULT_STRATEGY, 8, 9),
    (1, zlib.Z_DEFAULT_STRATEGY, 1, 9),
]


@gpu
@pytest.mark.parametrize("enc", ENCODERS, ids=["L%d-s%d-m%d-w%d" % e for e in ENCODERS])
def test_gpu_zlib_encoders(codec, enc):
    data = mixed(12, seed=enc[0] + 3 * enc[1])
    blob = zlib_member(data, *enc)
    check(codec, blob, data)
    assert launches(codec, blob) > one_warp_launches(codec)


@gpu
@pytest.mark.skipif(shutil.which("gzip") is None, reason="GNU gzip not on PATH")
@pytest.mark.parametrize("level", [1, 6, 9])
def test_gpu_gnu_gzip(codec, level):
    data = mixed(16, seed=10 + level)
    blob = gnu_gzip(data, level)
    check(codec, blob, data)
    assert launches(codec, blob) > one_warp_launches(codec)


@gpu
def test_gpu_python_gzip_with_a_file_name(codec):
    data = H.synth("fastq", 24 << 20, seed=7)
    blob = python_gzip(data)
    assert blob[3] & 8 and b"reads.fq\0" in blob[:40]
    check(codec, blob, data)
    assert launches(codec, blob) > one_warp_launches(codec)


# ---------------------------------------------------------------- 2. route


@gpu
def test_gpu_route_comes_from_the_input(codec):
    base = one_warp_launches(codec)
    data = H.synth("fastq", 4 << 20)
    plain = zlib_member(data)
    assert len(plain) - 18 > 2 * REGION
    assert launches(codec, plain) > base
    flushed = sync_flush_stream(data, [100000])
    assert launches(codec, flushed) == CHAIN_LAUNCHES
    assert device(codec, flushed) == data


@gpu
@pytest.mark.parametrize("extra", [0, 1], ids=["one-region", "one-region-plus-a-byte"])
def test_gpu_region_edge(codec, extra):
    base = one_warp_launches(codec)
    n = REGION + extra
    sizes = fill_sizes(n)
    payload = H.lcg_noise(sum(sizes))
    raw = stored_stream(payload, sizes)
    assert len(raw) == n and b"\x00\x00\xff\xff" not in raw
    blob = with_header(payload, raw, 0)
    check(codec, blob, payload)
    assert (launches(codec, blob) > base) == bool(extra)


# ---------------------------------------------------------------- 3. forced repair


def planted_stored(nreg):
    """stored blocks only; right after the block header at every region start, the first bytes of a zlib raw stream (a dynamic
    block header): every region's proposed start is false, so every region costs one repair round"""
    sizes = region_sizes(nreg)
    fake = zlib.compress(H.synth("fastq", 100000, seed=3), 6, wbits=-15)[:300]
    parts, at, k = [], 0, 0
    for n in sizes:
        if at % REGION == 0 and at:
            parts.append(fake + H.lcg_noise(n - len(fake)))
        else:
            parts.append(H.synth("sam", n, seed=k))
        at += n + 5
        k += 1
    payload = b"".join(parts)
    raw = stored_stream(payload, sizes)
    assert len(raw) == nreg * REGION
    return with_header(payload, raw, 0), payload


@gpu
def test_gpu_forced_repair(codec):
    nreg = 6
    blob, payload = planted_stored(nreg)
    assert blob.count(b"\x00\x00\xff\xff") == 0
    check(codec, blob, payload)
    # count 3, search 1, boundary pass: the first round and one repair per region after the first, batch 5
    assert launches(codec, blob) == 3 + 1 + nreg + 5


@gpu
def test_gpu_repair_round_limit(codec):
    nreg = ROUNDS + 4
    blob, payload = planted_stored(nreg)
    check(codec, blob, payload)
    # the first round and ROUNDS repairs, then one warp
    assert launches(codec, blob) == 3 + 1 + 1 + ROUNDS + 1


# ---------------------------------------------------------------- 4. merged regions


@gpu
@pytest.mark.parametrize("mib", [6, 24], ids=["within-the-chunk-cap", "beyond-the-chunk-cap"])
def test_gpu_fixed_huffman_merges_regions(codec, mib):
    data = H.synth("fastq", mib << 20, seed=mib)
    blob = zlib_member(data, 6, zlib.Z_FIXED)
    assert len(blob) > 2 * REGION
    assert (len(blob) < (4 << 20)) == (mib == 6)
    check(codec, blob, data, reference=mib == 6)


# ---------------------------------------------------------------- 5. a chance flush pattern


@gpu
def test_gpu_chance_flush_pattern(codec):
    noise = H.lcg_noise(300000)
    noise = noise[:150000] + b"\x00\x00\xff\xff" + noise[150000:]
    data = H.synth("fastq", 12 << 20, seed=4) + noise + H.synth("sam", 8 << 20, seed=5)
    blob = zlib_member(data, 6)
    assert b"\x00\x00\xff\xff" in blob and len(blob) > (4 << 20)
    check(codec, blob, data)
    # the flush-point count and chain, then the searched route: search, at least one boundary round, a batch
    assert launches(codec, blob) >= 3 + 8 + 1 + 1 + 5


# ---------------------------------------------------------------- 6. damage


@gpu
@pytest.mark.parametrize("enc", ["zlib", "gnu"])
def test_gpu_damage_gives_the_one_warp_outcome(codec, enc):
    if enc == "gnu" and shutil.which("gzip") is None:
        pytest.skip("GNU gzip not on PATH")
    data = H.synth("fastq", 1 << 20) + H.lcg_noise(100000) + H.synth("sam", 2 << 20)
    blob = zlib_member(data) if enc == "zlib" else gnu_gzip(data, 6)
    assert len(blob) > 2 * REGION and b"\x00\x00\xff\xff" not in blob
    rnd = random.Random(8 if enc == "zlib" else 9)
    seen = set()
    for _ in range(40):
        dmg = bytearray(blob)
        at = rnd.randrange(20, len(blob) - 8)
        dmg[at] ^= 1 << rnd.randrange(8)
        dmg = bytes(dmg)
        for flags in (0, B.VERIFY):
            want = outcome(one_warp, codec, dmg, flags)
            assert outcome(parallel, codec, dmg, flags) == want, (at, flags)
            assert outcome(device, codec, dmg, flags) == want, (at, flags)
            seen.add(want[0] if want[0] == "ok" else want[1])
    assert len(seen) >= 2
    bad_crc = bytearray(blob)
    bad_crc[-6] ^= 0x10
    bad_crc = bytes(bad_crc)
    assert outcome(parallel, codec, bad_crc, B.VERIFY) == ("err", B.E_CRC)
    assert outcome(device, codec, bad_crc, B.VERIFY) == ("err", B.E_CRC)
    assert parallel(codec, bad_crc) == data
    bad_isize = blob[:-4] + struct.pack("<I", len(data) - 1000)
    want = outcome(one_warp, codec, bad_isize)
    assert want[0] == "err"
    assert outcome(parallel, codec, bad_isize) == want
    assert outcome(device, codec, bad_isize, 0, len(data)) == want


@gpu
def test_gpu_no_space_before_any_search(codec):
    import torch
    data = H.synth("sam", 3 << 20)
    lib, n = codec.lib, ctypes.c_size_t()
    f = lib.b200bgzf_gzip_inflate_device
    d_out = torch.empty(16, dtype=torch.uint8, device="cuda")
    spent = []
    for blob in (zlib_member(data[:200000]), zlib_member(data)):
        d_in = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
        want = struct.unpack("<I", blob[-4:])[0]
        before = codec.launches()
        assert f(codec.h, d_in.data_ptr(), len(blob), d_out.data_ptr(), 10, ctypes.byref(n), 0, None) == B.E_NOSPACE
        assert n.value == want
        assert f(codec.h, d_in.data_ptr(), len(blob), None, 0, ctypes.byref(n), 0, None) == B.E_NOSPACE and n.value == want
        spent.append(codec.launches() - before)
    assert spent[0] == spent[1]          # the flush-point count only: no search for a member that cannot fit


# ---------------------------------------------------------------- 7. batches


@gpu
def test_gpu_batches_under_a_small_budget(tmp_path):
    noise = H.lcg_noise(256 * (24 << 10))
    data = b"".join(noise[i * (24 << 10) : (i + 1) * (24 << 10)] + H.synth("fastq", 8 << 10, seed=i) for i in range(256))
    (tmp_path / "a.gz").write_bytes(zlib_member(data, 6))
    script = (
        "import sys, zlib; sys.path[:0] = [%r, %r]\n"
        "import b200bgzf as B, test_gzip_parallel as T\n"
        "c = B.Codec(0)\n"
        "blob = open(%r + '/a.gz', 'rb').read()\n"
        "want = zlib.decompress(blob, 31)\n"
        "n = c.launches()\n"
        "assert T.parallel(c, blob, B.VERIFY) == want and T.device(c, blob) == want\n"
        "n = (c.launches() - n) // 2\n"
        "assert n >= 3 + 1 + 1 + 2 * 5, n\n"
        "print('ok')\n"
    ) % (os.path.dirname(B.__file__), os.path.dirname(os.path.abspath(__file__)), str(tmp_path))
    env = dict(os.environ, B200BGZF_GZIP_BUDGET=str(1 << 20))
    r = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr


# ---------------------------------------------------------------- 8. the applet


@gpu
def test_gpu_7gzip_applet(codec):
    data = H.synth("fastq", 64 << 20, seed=11)
    blob = gnu_gzip(data, 6) if shutil.which("gzip") else zlib_member(data)
    d = subprocess.run([GZIP_EXE, "-d"], input=blob, capture_output=True)
    assert d.returncode == 0 and d.stdout == data and b"1 done." in d.stderr


# ---------------------------------------------------------------- 9. large


@gpu
def test_gpu_one_gib_round_trip(codec):
    data = H.synth("fastq", 1 << 30)
    blob, want = zlib_member(data, 6), zlib.crc32(data)
    del data
    out = parallel(codec, blob, B.VERIFY)
    assert len(out) == 1 << 30 and zlib.crc32(out) == want
