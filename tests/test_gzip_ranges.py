"""Random access into one whole-stream gzip member through a checkpoint index: b200bgzf_gzip_index_host / _device and
b200bgzf_gzip_inflate_ranges_host / _device, and `7gzip --reindex` / `7gzip -d --offset`.  The oracles are Python's zlib and
the public index format of include/b200bgzf.h, parsed here on its own: every c_start must follow 00 00 ff ff, every chunk
CRC must match zlib's output, and at every access point zlib itself must restart from the stored window."""
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
import test_gzip_parallel as T

gpu = pytest.mark.gpu
GZIP_EXE = T.GZIP_EXE
MIB = 1 << 20


def parse_index(ix):
    """the index as the format in include/b200bgzf.h describes it (asserts its self-CRC and its size)"""
    assert ix[:8] == b"B2GZIX01"
    assert struct.unpack("<I", ix[-4:])[0] == zlib.crc32(ix[:-4])
    in_bytes, hdr_len, crc, isize, out_bytes, span, n, npts = struct.unpack_from("<QIIIQIII", ix, 8)
    chunks = [struct.unpack_from("<QQI", ix, 48 + 20 * k) for k in range(n)]
    points = [struct.unpack_from("<II", ix, 48 + 20 * n + 8 * p) for p in range(npts)]
    at, wins = 48 + 20 * n + 8 * npts, []
    for _, wl in points:
        wins.append(ix[at : at + wl])
        at += wl
    assert at + 4 == len(ix)
    return dict(in_bytes=in_bytes, hdr_len=hdr_len, crc=crc, isize=isize, out_bytes=out_bytes, span=span, chunks=chunks,
                points=[(c, w) for (c, _), w in zip(points, wins)])


def check_index(blob, ix, span, data=None, restart_sample=None):
    """every claim the index makes, against zlib"""
    data = zlib.decompress(blob, 31) if data is None else data
    x = parse_index(ix)
    assert (x["in_bytes"], x["out_bytes"], x["span"]) == (len(blob), len(data), span or MIB)
    assert (x["crc"], x["isize"]) == struct.unpack("<II", blob[-8:])
    ch = x["chunks"]
    assert ch[0][0] == x["hdr_len"] and ch[0][1] == 0
    ends = [u for _, u, _ in ch[1:]] + [len(data)]
    for k, (c, u, crc) in enumerate(ch):
        assert k == 0 or (blob[c - 4 : c] == b"\x00\x00\xff\xff" and c > ch[k - 1][0]), k
        assert zlib.crc32(data[u : ends[k]]) == crc, k
    want = [0]                                                   # access points: the spacing rule
    for k in range(1, len(ch)):
        if ch[k][1] - ch[want[-1]][1] >= (span or MIB):
            want.append(k)
    assert [c for c, _ in x["points"]] == want
    pts = x["points"] if restart_sample is None else random.Random(7).sample(x["points"], min(restart_sample, len(x["points"])))
    for k, win in x["points"]:
        u = ch[k][1]
        assert win == data[max(0, u - 32768) : u]
    for k, win in pts:                                           # zlib restarts at the point with the stored window
        c, u, _ = ch[k]
        d = zlib.decompressobj(-15, zdict=win) if win else zlib.decompressobj(-15)
        assert d.decompress(blob[c:]) == data[u:], k
    return x


def device_index(codec, blob, span=0):
    import torch
    d_in = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
    return codec.gzip_index_device(d_in.data_ptr(), len(blob), span)


def device_ranges(codec, blob, ix, ranges, flags=0):
    import torch
    d_in = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
    total = sum(e - b for b, e in ranges)
    d_out = torch.empty(max(total, 1), dtype=torch.uint8, device="cuda")
    got, off = codec.gzip_inflate_ranges_device(d_in.data_ptr(), len(blob), ix, ranges, d_out.data_ptr(), total, flags)
    return d_out[:got].cpu().numpy().tobytes(), off


def want_of(data, ranges):
    out, off = [], []
    at = 0
    for b, e in ranges:
        off.append(at)
        out.append(data[b:e])
        at += e - b
    return b"".join(out), off


def outcome(fn, *args):
    try:
        return ("ok", fn(*args))
    except B.B200BgzfError as e:
        return ("err", e.code)


@pytest.fixture(scope="module")
def codec():
    c = B.Codec(0)
    yield c
    c.close()


def index_inputs(codec):
    fq, sam = H.synth("fastq", 3 * MIB), H.synth("sam", 2 * MIB)
    rnd = random.Random(3)
    gaps = [rnd.choice([1, 7, 100, 2000, 20000, 40000, 130000, 300 << 10]) for _ in range(64)]
    mixed = H.synth("sam", MIB) + H.lcg_noise(300000) + H.synth("fastq", MIB)
    yield "primed", codec.container(B.CONTAINER_GZIP, fq, 6), fq
    yield "independent", codec.container(B.CONTAINER_GZIP, sam, 6, T.PARAM_INDEPENDENT), sam
    for mode, name in ((zlib.Z_SYNC_FLUSH, "sync"), (zlib.Z_FULL_FLUSH, "full")):
        for level in (1, 6):
            yield f"zlib-{name}-{level}", T.sync_flush_stream(mixed, gaps, level, mode, double_every=5), mixed
    small = H.synth("fastq", 400000)
    for flags in (4, 8, 16, 2, 4 | 8 | 16 | 2):
        yield f"header-{flags}", T.with_header(small, T.raw_deflate(small, 6, [50000]), flags, extra=b"AB\x02\x00xy", name=b"f.fq",
                                               comment=b"c" * 5000), small
    yield "x", codec.container(B.CONTAINER_GZIP, b"x", 6), b"x"
    yield "zeros", codec.container(B.CONTAINER_GZIP, bytes(2 * MIB), 6), bytes(2 * MIB)
    yield "plain-zeros", zlib.compress(bytes(3 * MIB), 6, wbits=31), bytes(3 * MIB)     # no flush point: one chunk
    yield "plain-small", zlib.compress(small, 6, wbits=31), small


# ---------------------------------------------------------------- 1. the index against zlib


@gpu
def test_gpu_index_against_zlib(codec):
    for name, blob, data in index_inputs(codec):
        for span in (32768, 0, 2 * len(data) + MIB):
            ix = codec.gzip_index(blob, span)
            x = check_index(blob, ix, span, data)
            assert ix == device_index(codec, blob, span) == codec.gzip_index(blob, span), (name, span)
            if span > len(data):
                assert len(x["points"]) == 1, name
            elif span == 32768:                                  # (a chunk of 48 KiB or more is a point of its own)
                assert len(x["points"]) > {"primed": 60, "zlib-sync-6": 10}.get(name, 0), name
        if name in ("x", "plain-zeros", "plain-small"):
            assert len(parse_index(ix)["chunks"]) == 1, name


@gpu
def test_gpu_index_refusals(codec):
    noise = H.lcg_noise(8 * MIB)
    plain = zlib.compress(noise, 6, wbits=31)
    assert len(plain) > 4 * MIB
    a, b = H.synth("fastq", 300000), H.synth("sam", 300000)
    two = codec.container(B.CONTAINER_GZIP, a, 6) + codec.container(B.CONTAINER_GZIP, b, 6)
    bad_isize = bytearray(codec.container(B.CONTAINER_GZIP, a, 6))
    bad_isize[-1] ^= 0x01
    for blob in (plain, two, T.sync_flush_stream(a, [50000]) + T.sync_flush_stream(b, [50000]), bytes(bad_isize), H.lcg_noise(100000)):
        assert outcome(codec.gzip_index, blob)[1] == B.E_FORMAT
        assert outcome(device_index, codec, blob)[1] == B.E_FORMAT
    good = codec.container(B.CONTAINER_GZIP, a, 6)
    lib, n = codec.lib, ctypes.c_size_t()
    assert outcome(codec.gzip_index, good, 1000) == ("err", B.E_ARG)
    assert outcome(codec.gzip_index, good, 32767) == ("err", B.E_ARG)
    f = lib.b200bgzf_gzip_index_host
    assert f(None, B._addr(good), len(good), 0, None, 0, ctypes.byref(n)) == B.E_ARG
    assert f(codec.h, None, len(good), 0, None, 0, ctypes.byref(n)) == B.E_ARG
    assert f(codec.h, B._addr(good), len(good), 0, None, 0, None) == B.E_ARG
    assert f(codec.h, B._addr(good), len(good), 0, None, 0, ctypes.byref(n)) == B.E_NOSPACE
    ix = codec.gzip_index(good)
    assert n.value == len(ix)
    buf = ctypes.create_string_buffer(len(ix) - 1)
    assert f(codec.h, B._addr(good), len(good), 0, buf, len(ix) - 1, ctypes.byref(n)) == B.E_NOSPACE and n.value == len(ix)


# ---------------------------------------------------------------- 2. ranges against zlib


def range_cases(x, rnd, nrandom=300):
    total = x["out_bytes"]
    us = [u for _, u, _ in x["chunks"]]
    ps = [x["chunks"][c][1] for c, _ in x["points"]]
    rs = []
    for _ in range(nrandom):
        b = rnd.randrange(total + 1)
        rs.append((b, min(total, b + rnd.choice([0, 1, 100, 5000, 70000, 400000]))))
    for u in rnd.sample(us, min(60, len(us))):
        rs += [(max(0, u - 1), min(total, u + 1)), (u, u), (u, min(total, u + 5000))]
    for u in ps:
        rs += [(max(0, u - 5), min(total, u + 5)), (max(0, u - 40000), u)]
    rs += [(total - 10, total), (total, total), (0, total), (1000, 9000), (1000, 9000), (5000, 200000), (0, 1)]
    rnd.shuffle(rs)
    return rs


@gpu
@pytest.mark.parametrize("span", [32768, 0])
def test_gpu_ranges_against_zlib(codec, span):
    rnd = random.Random(11 + span)
    data = H.synth("fastq", 6 * MIB) + H.synth("sam", 2 * MIB)
    rnd_gaps = [rnd.choice([100, 2000, 20000, 40000, 130000]) for _ in range(40)]
    for blob in (codec.container(B.CONTAINER_GZIP, data, 6), T.sync_flush_stream(data, rnd_gaps, 6, double_every=7)):
        ix = codec.gzip_index(blob, span)
        x = parse_index(ix)
        rs = range_cases(x, rnd)
        want, woff = want_of(data, rs)
        for flags in (0, B.VERIFY):
            got, off = codec.gzip_inflate_ranges(blob, ix, rs, flags)
            assert got == want and off == woff
            dgot, doff = device_ranges(codec, blob, ix, rs, flags)
            assert dgot == want and doff == woff
        for r in rs[:40]:                                        # one range per call
            assert codec.gzip_inflate_ranges(blob, ix, [r])[0] == data[r[0] : r[1]]
        assert codec.gzip_inflate_ranges(blob, ix, []) == (b"", [])


# ---------------------------------------------------------------- 3. batches under a small budget


@gpu
def test_gpu_ranges_batch_under_a_small_budget(tmp_path):
    data = H.synth("fastq", 6 * MIB) + (H.lcg_noise(30 << 10) * 40)
    c = B.Codec(0)
    (tmp_path / "a.gz").write_bytes(c.container(B.CONTAINER_GZIP, data, 6))
    (tmp_path / "b.gz").write_bytes(T.sync_flush_stream(data, [7000, 300, 45000], 6))
    c.close()
    script = (
        "import sys, random, zlib; sys.path[:0] = [%r, %r]\n"
        "import b200bgzf as B, test_gzip_ranges as G\n"
        "c = B.Codec(0)\n"
        "for f in ('a.gz', 'b.gz'):\n"
        "    blob = open(%r + '/' + f, 'rb').read()\n"
        "    data = zlib.decompress(blob, 31)\n"
        "    for span in (32768, 0):\n"
        "        ix = c.gzip_index(blob, span)\n"
        "        x = G.check_index(blob, ix, span, data, restart_sample=4)\n"
        "        rs = G.range_cases(x, random.Random(5), 200) + [(100, 3 * (1 << 20)), (len(data) - 2500000, len(data))]\n"
        "        want, woff = G.want_of(data, rs)\n"
        "        assert c.gzip_inflate_ranges(blob, ix, rs, B.VERIFY) == (want, woff)\n"
        "        assert G.device_ranges(c, blob, ix, rs) == (want, woff)\n"
        "print('ok')\n"
    ) % (os.path.dirname(B.__file__), os.path.dirname(os.path.abspath(__file__)), str(tmp_path))
    env = dict(os.environ, B200BGZF_GZIP_BUDGET=str(MIB))
    r = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr


# ---------------------------------------------------------------- 4. locality


def touched_bytes(x, in_bytes, beg, end):
    """[first, last) of the compressed bytes a range's run reads: from its access point to the end of its last chunk"""
    us = [u for _, u, _ in x["chunks"]]
    f = max(k for k, u in enumerate(us) if u <= beg)
    last = max(k for k, u in enumerate(us) if u <= end - 1)
    p = max(c for c, _ in x["points"] if c <= f)
    stop = x["chunks"][last + 1][0] if last + 1 < len(us) else in_bytes - 8
    return x["chunks"][p][0], stop


@gpu
def test_gpu_only_touched_runs_are_read(codec):
    data = H.synth("fastq", 8 * MIB)
    blob = codec.container(B.CONTAINER_GZIP, data, 6)
    ix = codec.gzip_index(blob, 32768)
    x = parse_index(ix)
    rs = [(1000, 5000), (3 * MIB + 77, 3 * MIB + 90000), (7 * MIB, 7 * MIB + 1)]
    spans = [touched_bytes(x, len(blob), b, e) for b, e in rs]
    keep = bytearray(len(blob))
    for lo, hi in spans:
        keep[lo:hi] = blob[lo:hi]
    keep[-8:] = blob[-8:]
    want, woff = want_of(data, rs)
    assert codec.gzip_inflate_ranges(bytes(keep), ix, rs, B.VERIFY) == (want, woff)
    rnd = random.Random(9)
    inside = [i for lo, hi in spans for i in range(lo, hi)]
    outside = [i for i in range(len(blob) - 8) if not keep[i] and blob[i]]
    for _ in range(20):                                          # a flip in an untouched chunk changes nothing
        dmg = bytearray(blob)
        dmg[rnd.choice(outside)] ^= 1 << rnd.randrange(8)
        assert codec.gzip_inflate_ranges(bytes(dmg), ix, rs, B.VERIFY) == (want, woff)
    errors = 0
    for _ in range(40):                                          # a flip in a touched chunk: an error, never wrong bytes
        dmg = bytearray(blob)
        dmg[rnd.choice(inside)] ^= 1 << rnd.randrange(8)
        got = outcome(codec.gzip_inflate_ranges, bytes(dmg), ix, rs, B.VERIFY)
        assert got == ("ok", (want, woff)) or got[1] in (B.E_FORMAT, B.E_CRC), got[:1]
        errors += got[0] == "err"
    assert errors >= 30


# ---------------------------------------------------------------- 5. refusals


@gpu
def test_gpu_range_refusals(codec):
    import torch
    data = H.synth("sam", 3 * MIB)
    blob = codec.container(B.CONTAINER_GZIP, data, 6)
    other = codec.container(B.CONTAINER_GZIP, data[:-1] + b"!", 6)
    ix = codec.gzip_index(blob, 32768)
    lib, n = codec.lib, ctypes.c_size_t()
    rs = (B.Range * 2)(B.Range(10, 20000), B.Range(MIB, MIB + 5))
    out = ctypes.create_string_buffer(20000)
    f = lib.b200bgzf_gzip_inflate_ranges_host
    flipped = bytearray(ix)
    flipped[len(ix) // 2] ^= 4
    resealed = bytearray(ix)                                      # chunks out of order, self-CRC made valid again
    resealed[48:68], resealed[68:88] = ix[68:88], ix[48:68]
    resealed[-4:] = struct.pack("<I", zlib.crc32(bytes(resealed[:-4])))
    grown = ix[:-4] + b"\0" + struct.pack("<I", zlib.crc32(ix[:-4] + b"\0"))
    other_ix = codec.gzip_index(other, 32768)
    before = codec.launches()
    for bad in (other_ix, ix[:-1], ix[: len(ix) // 2], bytes(flipped), bytes(resealed), grown, b"", b"B2GZIX01"):
        assert f(codec.h, B._addr(blob), len(blob), B._addr(bad) if bad else None, len(bad), rs, 2, out, 20000, ctypes.byref(n), None, 0) \
            in ((B.E_FORMAT,) if bad else (B.E_ARG,))
        assert codec.launches() == before
    assert f(codec.h, B._addr(blob), len(blob) - 1, B._addr(ix), len(ix), rs, 2, out, 20000, ctypes.byref(n), None, 0) == B.E_FORMAT
    assert codec.launches() == before
    off = (ctypes.c_uint64 * 2)()
    assert f(codec.h, B._addr(blob), len(blob), B._addr(ix), len(ix), rs, 2, out, 19994, ctypes.byref(n), off, 0) == B.E_NOSPACE
    assert n.value == 19995 and list(off) == [0, 19990] and codec.launches() == before
    assert f(codec.h, B._addr(blob), len(blob), B._addr(ix), len(ix), rs, 2, None, 0, ctypes.byref(n), None, 0) == B.E_NOSPACE
    for bad in ((5, 4), (0, len(data) + 1), (len(data) + 1, len(data) + 1)):
        br = (B.Range * 1)(B.Range(*bad))
        assert f(codec.h, B._addr(blob), len(blob), B._addr(ix), len(ix), br, 1, out, 20000, ctypes.byref(n), None, 0) == B.E_ARG
    args = [codec.h, B._addr(blob), len(blob), B._addr(ix), len(ix), rs, 2, out, 20000, ctypes.byref(n), None, 0]
    for k in (0, 1, 3, 5, 9):
        a = list(args)
        a[k] = None
        assert f(*a) == B.E_ARG, k
    assert f(*(args[:-1] + [B.RANGE_VOFFSET])) == B.E_ARG
    assert codec.launches() == before
    assert f(*args) == 0 and n.value == 19995 and out.raw[:19995] == data[10:20000] + data[MIB : MIB + 5]
    d_in = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
    d_out = torch.empty(20000, dtype=torch.uint8, device="cuda")
    g = lib.b200bgzf_gzip_inflate_ranges_device
    for bad in (other_ix, ix[:-1], bytes(flipped)):
        assert g(codec.h, d_in.data_ptr(), len(blob), B._addr(bad), len(bad), rs, 2, d_out.data_ptr(), 20000, ctypes.byref(n), None, 0, None) == B.E_FORMAT
    assert g(codec.h, d_in.data_ptr(), len(blob), B._addr(ix), len(ix), rs, 2, d_out.data_ptr(), 100, ctypes.byref(n), None, 0, None) == B.E_NOSPACE
    assert n.value == 19995
    assert g(codec.h, d_in.data_ptr(), len(blob), B._addr(ix), len(ix), rs, 2, d_out.data_ptr(), 20000, ctypes.byref(n), None,
             B.RANGE_VOFFSET, None) == B.E_ARG


# ---------------------------------------------------------------- 6. the applet


def test_7gzip_index_usage():
    """command lines refused before any GPU work"""
    for args in (["-d", "--offset=5"], ["--reindex"], ["--index=/dev/null"], ["-d", "--index=/dev/null"],
                 ["--reindex", "--index=/dev/null", "-d"], ["-d", "--offset=5", "--index=/dev/null", "--gzi=/dev/null"],
                 ["-d", "--offset=x", "--index=/dev/null"], ["-l6", "--offset=5", "--index=/dev/null"]):
        r = subprocess.run([GZIP_EXE] + args, input=b"", capture_output=True)
        assert r.returncode != 0 and b"Usage" in r.stderr, args
    r = subprocess.run([B.APPLET_PATH, "-d", "--offset=5", "--index=/dev/null"], input=b"", capture_output=True)
    assert r.returncode != 0 and b"Usage" in r.stderr                # --index belongs to 7gzip


@gpu
def test_gpu_7gzip_reindex_and_offset(codec, tmp_path):
    data = H.synth("fastq", 64 * MIB)
    gz, idx = tmp_path / "in.gz", tmp_path / "in.gzx"
    gz.write_bytes(codec.container(B.CONTAINER_GZIP, data, 6))
    with open(gz, "rb") as f:
        r = subprocess.run([GZIP_EXE, "--reindex", f"--index={idx}"], stdin=f, capture_output=True)
    assert r.returncode == 0 and r.stdout == b"", r.stderr
    assert idx.read_bytes() == codec.gzip_index(gz.read_bytes())
    for off, size in ((0, 100), (12345678, 3 * MIB + 5), (len(data) - 10, 1000), (len(data), 5), (33 * MIB, None)):
        with open(gz, "rb") as f:
            r = subprocess.run([GZIP_EXE, "-d", f"--offset={off}", f"--index={idx}"] + ([] if size is None else [f"--size={size}"]),
                               stdin=f, capture_output=True)
        assert r.returncode == 0 and r.stdout == data[off : None if size is None else off + size], (off, size, r.stderr)
    bad = [["-d", f"--offset={len(data) + 1}", f"--index={idx}"], ["-d", "--offset=5", f"--index={tmp_path / 'missing'}"],
           ["-d", "--offset=5", f"--index={gz}"]]
    for args in bad:
        with open(gz, "rb") as f:
            r = subprocess.run([GZIP_EXE] + args, stdin=f, capture_output=True)
        assert r.returncode != 0 and r.stdout == b"" and r.stderr, args
    other = tmp_path / "other.gz"
    other.write_bytes(codec.container(B.CONTAINER_GZIP, data[: 8 * MIB], 6))
    with open(other, "rb") as f:
        r = subprocess.run([GZIP_EXE, "-d", "--offset=5", "--size=10", f"--index={idx}"], stdin=f, capture_output=True)
    assert r.returncode != 0 and r.stdout == b""
    r = subprocess.run([GZIP_EXE, "--reindex", f"--index={tmp_path / 'x.gzx'}"], input=zlib.compress(H.lcg_noise(8 * MIB), 6, wbits=31),
                       capture_output=True)
    assert r.returncode != 0 and not (tmp_path / "x.gzx").exists()
    d = subprocess.run([GZIP_EXE, "-d"], stdin=open(gz, "rb"), capture_output=True)   # the whole-file command line is unchanged
    assert d.returncode == 0 and d.stdout == data


# ---------------------------------------------------------------- 7. large


@gpu
def test_gpu_one_gib_index_and_1000_ranges(codec):
    data = H.synth("fastq", 1 << 30)
    blob = codec.container(B.CONTAINER_GZIP, data, 6)
    ix = codec.gzip_index(blob)
    x = parse_index(ix)
    us = [u for _, u, _ in x["chunks"]] + [len(data)]
    assert x["out_bytes"] == len(data) and len(x["points"]) > 900
    for k in random.Random(1).sample(range(len(x["chunks"])), 500):
        assert zlib.crc32(data[us[k] : us[k + 1]]) == x["chunks"][k][2]
    rnd = random.Random(2)
    rs = []
    for _ in range(1000):
        b = rnd.randrange(len(data))
        rs.append((b, min(len(data), b + rnd.choice([1, 4096, 65536, MIB]))))
    got, off = codec.gzip_inflate_ranges(blob, ix, rs, B.VERIFY)
    for (b, e), o in zip(rs, off):
        assert zlib.crc32(got[o : o + e - b]) == zlib.crc32(data[b:e])
