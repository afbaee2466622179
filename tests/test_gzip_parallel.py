"""Whole-stream gzip decoded in parallel between its byte-aligned flush points: b200bgzf_container_inflate_host(GZIP) and
b200bgzf_gzip_inflate_device.  Every stream is checked against zlib and, where one warp finishes in seconds, against the
one-warp path (b200bgzf_inflate_units_host over the one-unit list of b200bgzf_container_units), whose bytes or error code
the parallel path must reproduce exactly."""
import ctypes
import os
import random
import struct
import subprocess
import sys
import zlib

import pytest

import b200bgzf as B
import helpers as H

gpu = pytest.mark.gpu
PARAM_INDEPENDENT = 0x20000000
GZIP_EXE = os.path.join(os.path.dirname(B.APPLET_PATH), "7gzip")


def sync_flush_stream(data, gaps, level=6, mode=zlib.Z_SYNC_FLUSH, wbits=31, double_every=0):
    """zlib stream of `data` with a flush after every gap (cycling through `gaps`); every `double_every`-th flush is given
    twice in a row (an empty chunk between two flush points)"""
    z = zlib.compressobj(level, zlib.DEFLATED, wbits)
    out, at, i = [], 0, 0
    while at < len(data):
        g = gaps[i % len(gaps)]
        out.append(z.compress(data[at : at + g]))
        out.append(z.flush(mode))
        if double_every and i % double_every == 0:
            out.append(z.flush(mode))
        at += g
        i += 1
    out.append(z.flush())
    return b"".join(out)


def with_header(data, raw, flags, extra=b"", name=b"", comment=b""):
    """a gzip member around raw DEFLATE data with a hand-built header (FEXTRA / FNAME / FCOMMENT / FHCRC)"""
    h = bytes([0x1F, 0x8B, 8, flags, 0, 0, 0, 0, 0, 3])
    if flags & 4:
        h += struct.pack("<H", len(extra)) + extra
    if flags & 8:
        h += name + b"\0"
    if flags & 16:
        h += comment + b"\0"
    if flags & 2:
        h += struct.pack("<H", zlib.crc32(h) & 0xFFFF)
    return h + raw + struct.pack("<II", zlib.crc32(data), len(data) & 0xFFFFFFFF)


def raw_deflate(data, level=6, gaps=None, mode=zlib.Z_SYNC_FLUSH):
    return sync_flush_stream(data, gaps, level, mode, wbits=-15) if gaps else zlib.compress(data, level, wbits=-15)


def outcome(fn, *args):
    try:
        return ("ok", fn(*args))
    except B.B200BgzfError as e:
        return ("err", e.code)


def one_warp(codec, blob, flags=0):
    units, total = B.container_units(B.CONTAINER_GZIP, blob)
    return codec.inflate_units(blob, units, total, flags)


def parallel(codec, blob, flags=0):
    return codec.container_inflate(B.CONTAINER_GZIP, blob, flags)


def device(codec, blob, flags=0, cap=None):
    import torch
    d_in = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
    n = struct.unpack("<I", blob[-4:])[0] if cap is None else cap
    d_out = torch.empty(max(n, 1), dtype=torch.uint8, device="cuda")
    got = codec.gzip_inflate_device(d_in.data_ptr(), len(blob), d_out.data_ptr(), n, flags)
    return d_out[:got].cpu().numpy().tobytes()


def check(codec, blob, data, reference=True):
    assert zlib.decompress(blob, 31) == data
    assert parallel(codec, blob) == data
    assert device(codec, blob) == data
    if reference:
        assert one_warp(codec, blob) == data


@pytest.fixture(scope="module")
def codec():
    c = B.Codec(0)
    yield c
    c.close()


def inputs():
    return {
        "fastq": H.synth("fastq", 3 << 20),
        "sam": H.synth("sam", 3 << 20),
        "noise": H.lcg_noise(1 << 20),
        "x": b"x",
        "zeros": bytes(2 << 20),
    }


# ---------------------------------------------------------------- 1. our own files


@gpu
@pytest.mark.parametrize("param", [0, PARAM_INDEPENDENT], ids=["primed", "independent"])
def test_gpu_own_files(codec, param):
    for name, data in inputs().items():
        blob = codec.container(B.CONTAINER_GZIP, data, 6, param)
        check(codec, blob, data)
        assert parallel(codec, blob, B.VERIFY) == data and device(codec, blob, B.VERIFY) == data, name


@gpu
@pytest.mark.parametrize("param", [0, PARAM_INDEPENDENT], ids=["primed", "independent"])
def test_gpu_own_file_64mib(codec, param):
    data = H.synth("fastq", 64 << 20)
    blob = codec.container(B.CONTAINER_GZIP, data, 6, param)
    check(codec, blob, data, reference=False)


# ---------------------------------------------------------------- 2. zlib flush streams


@gpu
@pytest.mark.parametrize("level", [0, 1, 6, 9])
@pytest.mark.parametrize("mode", [zlib.Z_SYNC_FLUSH, zlib.Z_FULL_FLUSH], ids=["sync", "full"])
def test_gpu_zlib_flush_streams(codec, level, mode):
    rnd = random.Random(level * 10 + mode)
    data = H.synth("sam", 1 << 20) + H.lcg_noise(300000) + H.synth("fastq", 1 << 20)
    # gaps of 1 B .. 300 KiB: chunks far shorter than 32 KiB (windows over several chunks), consecutive flushes
    gaps = [rnd.choice([1, 7, 100, 2000, 20000, 40000, 130000, 300 << 10]) for _ in range(64)]
    blob = sync_flush_stream(data, gaps, level, mode, double_every=5)
    check(codec, blob, data)


@gpu
@pytest.mark.parametrize("flags", [4, 8, 16, 2, 4 | 8 | 16 | 2])
def test_gpu_hand_built_headers(codec, flags):
    data = H.synth("fastq", 500000)
    blob = with_header(data, raw_deflate(data, 6, [50000]), flags, extra=b"AB\x02\x00xy", name=b"file.fq", comment=b"c" * 5000)
    check(codec, blob, data)


# ---------------------------------------------------------------- 3. the worst-case dependency chain


@gpu
def test_gpu_worst_case_chain(codec):
    """30 KiB of noise repeated, a sync flush every 40 KiB: every byte of every chunk after the first refers before its
    chunk, so the markers form one run over all chunks"""
    data = (H.lcg_noise(30 << 10) * ((64 << 20) // (30 << 10) + 1))[: 64 << 20]
    blob = sync_flush_stream(data, [40 << 10], 6)
    check(codec, blob, data, reference=False)
    small = blob if len(data) <= (4 << 20) else sync_flush_stream(data[: 4 << 20], [40 << 10], 6)
    assert one_warp(codec, small) == parallel(codec, small) == data[: 4 << 20]


# ---------------------------------------------------------------- 4. false candidates


@gpu
@pytest.mark.parametrize("level", [0, 6])
def test_gpu_payload_dense_in_flush_patterns(codec, level):
    rnd = random.Random(4 + level)
    parts = []
    for _ in range(400):
        parts.append(b"\x00\x00\xff\xff" * rnd.randrange(1, 200))
        parts.append(H.synth("fastq", rnd.randrange(10, 3000), seed=rnd.randrange(1 << 30)))
    data = b"".join(parts)
    blob = sync_flush_stream(data, [70000, 1000, 33000], level)
    check(codec, blob, data)


@gpu
def test_gpu_planted_candidate_decodes_long(codec):
    """a stored block whose bytes are 00 00 ff ff and then a valid DEFLATE stream of 40 MiB of zeros: the candidate inside it
    decodes a long chunk that is not on the chain"""
    plant = b"\x00\x00\xff\xff" + zlib.compress(bytes(40 << 20), 9, wbits=-15)
    data = H.synth("sam", 200000) + plant + H.synth("fastq", 200000)
    blob = sync_flush_stream(data, [100000], 0)          # level 0: the plant stays in stored blocks
    check(codec, blob, data)


# ---------------------------------------------------------------- 5. fallback


@gpu
def test_gpu_fallback_streams(codec):
    data = H.synth("fastq", 2 << 20)
    plain = zlib.compress(data, 6, wbits=31)              # no flush point
    check(codec, plain, data)
    ref = open(os.path.join(H.GOLDEN, "containers", "ref.gz"), "rb").read()
    assert b"\x00\x00\xff\xff" not in ref
    assert parallel(codec, ref) == one_warp(codec, ref) == zlib.decompress(ref, 31)


@gpu
def test_gpu_concatenated_members(codec):
    a, b = H.synth("fastq", 300000), H.synth("sam", 300000)
    for blob in (sync_flush_stream(a, [50000]) + sync_flush_stream(b, [50000]),
                 codec.container(B.CONTAINER_GZIP, a, 6) + codec.container(B.CONTAINER_GZIP, b, 6)):
        for flags in (0, B.VERIFY):
            assert outcome(parallel, codec, blob, flags) == outcome(one_warp, codec, blob, flags)


# ---------------------------------------------------------------- 6. damage


@gpu
def test_gpu_damage_gives_the_one_warp_outcome(codec):
    data = H.synth("fastq", 600000) + H.lcg_noise(100000) + H.synth("sam", 350000)
    blob = sync_flush_stream(data, [20000, 90000, 3000], 6)
    rnd = random.Random(6)
    seen = set()
    for _ in range(40):
        dmg = bytearray(blob)
        at = rnd.randrange(10, len(blob) - 8)
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
    assert outcome(parallel, codec, bytes(bad_crc), B.VERIFY) == ("err", B.E_CRC)
    assert outcome(device, codec, bytes(bad_crc), B.VERIFY) == ("err", B.E_CRC)
    assert parallel(codec, bytes(bad_crc)) == data
    for cut in (len(blob) // 2, len(blob) - 9):
        assert outcome(parallel, codec, blob[:cut])[0] == "err"


# ---------------------------------------------------------------- 7. batches


@gpu
def test_gpu_batches_under_a_small_budget(tmp_path):
    data = H.synth("fastq", 6 << 20) + (H.lcg_noise(30 << 10) * 40)
    primed = B.Codec(0).container(B.CONTAINER_GZIP, data, 6)
    flushed = sync_flush_stream(data, [7000, 300, 45000], 6)
    (tmp_path / "a.gz").write_bytes(primed)
    (tmp_path / "b.gz").write_bytes(flushed)
    script = (
        "import sys, zlib; sys.path[:0] = [%r, %r]\n"
        "import b200bgzf as B, test_gzip_parallel as T\n"
        "c = B.Codec(0)\n"
        "for f in ('a.gz', 'b.gz'):\n"
        "    blob = open(%r + '/' + f, 'rb').read()\n"
        "    want = zlib.decompress(blob, 31)\n"
        "    assert T.parallel(c, blob, B.VERIFY) == want and T.device(c, blob) == want\n"
        "print('ok')\n"
    ) % (os.path.dirname(B.__file__), os.path.dirname(os.path.abspath(__file__)), str(tmp_path))
    env = dict(os.environ, B200BGZF_GZIP_BUDGET=str(1 << 20))
    r = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr


# ---------------------------------------------------------------- 8. argument errors


@gpu
def test_gpu_argument_errors(codec):
    import torch
    data = H.synth("sam", 400000)
    blob = sync_flush_stream(data, [30000])
    d_in = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
    d_out = torch.empty(len(data), dtype=torch.uint8, device="cuda")
    lib, n = codec.lib, ctypes.c_size_t()
    f = lib.b200bgzf_gzip_inflate_device
    assert f(codec.h, d_in.data_ptr(), len(blob), d_out.data_ptr(), len(data) - 1, ctypes.byref(n), 0, None) == B.E_NOSPACE
    assert n.value == len(data)
    assert f(codec.h, d_in.data_ptr(), len(blob), None, 0, ctypes.byref(n), 0, None) == B.E_NOSPACE and n.value == len(data)
    plain = zlib.compress(data, 6, wbits=31)            # (the one-warp route sizes the same way)
    p_in = torch.frombuffer(bytearray(plain), dtype=torch.uint8).cuda()
    assert f(codec.h, p_in.data_ptr(), len(plain), d_out.data_ptr(), 10, ctypes.byref(n), 0, None) == B.E_NOSPACE and n.value == len(data)
    assert f(None, d_in.data_ptr(), len(blob), d_out.data_ptr(), len(data), ctypes.byref(n), 0, None) == B.E_ARG
    assert f(codec.h, None, len(blob), d_out.data_ptr(), len(data), ctypes.byref(n), 0, None) == B.E_ARG
    assert f(codec.h, d_in.data_ptr(), len(blob), d_out.data_ptr(), len(data), None, 0, None) == B.E_ARG
    assert f(codec.h, d_in.data_ptr(), 0, d_out.data_ptr(), len(data), ctypes.byref(n), 0, None) != 0
    junk = torch.frombuffer(bytearray(H.lcg_noise(100000)), dtype=torch.uint8).cuda()
    assert f(codec.h, junk.data_ptr(), 100000, d_out.data_ptr(), len(data), ctypes.byref(n), 0, None) == B.E_FORMAT
    assert f(codec.h, d_in.data_ptr(), len(blob), d_out.data_ptr(), len(data), ctypes.byref(n), 0, None) == 0
    assert n.value == len(data) and d_out.cpu().numpy().tobytes() == data


# ---------------------------------------------------------------- 9. the applet


@gpu
def test_gpu_7gzip_applet(codec):
    data = H.synth("fastq", 64 << 20)
    small = H.synth("sam", 3 << 20)
    for blob, want in ((codec.container(B.CONTAINER_GZIP, data, 6), data), (sync_flush_stream(small, [128 << 10]), small)):
        d = subprocess.run([GZIP_EXE, "-d"], input=blob, capture_output=True)
        assert d.returncode == 0 and d.stdout == want and b"1 done." in d.stderr


# ---------------------------------------------------------------- 10. large


@gpu
def test_gpu_one_gib_round_trip(codec):
    data = H.synth("fastq", 1 << 30)
    blob = codec.container(B.CONTAINER_GZIP, data, 6)
    out = parallel(codec, blob, B.VERIFY)
    assert len(out) == len(data) and zlib.crc32(out) == zlib.crc32(data)


@gpu
def test_gpu_path_choice_comes_from_the_input(codec):
    """a member with flush points goes through the chunked decode (count, chain and batch launches); one without them
    through the one-warp kernel"""
    import torch
    data = H.synth("fastq", 1 << 20)
    for blob, chunked in ((sync_flush_stream(data, [100000]), True), (zlib.compress(data, 6, wbits=31), False)):
        d_in = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
        d_out = torch.empty(len(data), dtype=torch.uint8, device="cuda")
        before = codec.launches()
        assert codec.gzip_inflate_device(d_in.data_ptr(), len(blob), d_out.data_ptr(), len(data)) == len(data)
        assert d_out.cpu().numpy().tobytes() == data
        assert (codec.launches() - before >= 16) == chunked
