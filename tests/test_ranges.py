"""Random access: b200bgzf_index_host / b200bgzf_gzi_parse (CPU), b200bgzf_inflate_ranges_host / _device and the applet's
-d --offset / --reindex.  The truth for every range is data[beg:end] of the original input (or of H.gunzip of a golden stream)."""
import ctypes
import os
import random
import struct
import subprocess
import sys

import pytest

import b200bgzf
import helpers as H

gpu = pytest.mark.gpu
APPLET = b200bgzf.APPLET_PATH


def _slices(data, ranges):
    out, offs = bytearray(), []
    for b, e in ranges:
        offs.append(len(out))
        out += data[b:e]
    return bytes(out), offs


def _cend(c, n_in, m):
    return c[m + 1] if m + 1 < len(c) else n_in


# ---------------------------------------------------------------- CPU: the index helpers and the command line


@pytest.mark.parametrize("pairs", [([0], [0]), ([0, 100], [0, 65280]), ([0, 17, 4000, 9000, 9028], [0, 65280, 130560, 140000, 140000])])
def test_gzi_parse_inverts_gzi_format(pairs):
    c, u = pairs
    assert b200bgzf.gzi_parse(b200bgzf.gzi_format(c, u)) == (c, u)


def test_gzi_parse_refuses_malformed_files():
    good = b200bgzf.gzi_format([0, 100, 200], [0, 65280, 130560])
    bad = {
        "truncated": good[:-1],
        "short": good[:5],
        "miscounted": struct.pack("<Q", 3) + good[8:],
        "descending compressed": struct.pack("<QQQQQ", 2, 200, 65280, 100, 130560),
        "descending uncompressed": struct.pack("<QQQQQ", 2, 100, 130560, 200, 65280),
        "repeated first entry": struct.pack("<QQQ", 1, 0, 0),
    }
    for what, blob in bad.items():
        with pytest.raises(b200bgzf.B200BgzfError) as e:
            b200bgzf.gzi_parse(blob)
        assert e.value.code == b200bgzf.E_FORMAT, what


def _emulated_streams():
    for kind, level, n, eof in (("fastq", 6, 7 * H.BLOCK + 123, True), ("sam", 1, 5 * H.BLOCK, True), ("sam", 6, 3 * H.BLOCK + 9, False)):
        data = H.synth(kind, n)
        yield f"{kind}-L{level}", data, H.emul_stream(data, level, eof=eof)


def _golden_streams():
    for name in sorted(os.listdir(H.GOLDEN)):
        if name.startswith("ref_") and name.endswith(".bgz"):
            blob = open(os.path.join(H.GOLDEN, name), "rb").read()
            yield name, H.gunzip(blob), blob


def test_index_agrees_with_the_header_walk_and_the_gzi():
    seen = 0
    for name, data, stream in list(_emulated_streams()) + list(_golden_streams()):
        c, u = b200bgzf.index(stream)
        ms = H.members(stream)
        assert c == [m[0] for m in ms], name
        pos, want_u = 0, []
        for m in ms:
            want_u.append(pos)
            pos += m[2]
        assert u == want_u and pos == len(data), name
        # the .gzi lists the members that carry data, the first one implicitly
        keep = [(cc, uu) for k, (cc, uu) in enumerate(zip(c, u)) if ms[k][2]]
        assert b200bgzf.gzi_format([k[0] for k in keep], [k[1] for k in keep]) == H.gzi_of(stream), name
        seen += 1
    assert seen >= 9


def test_index_refuses_a_stream_that_is_not_bgzf():
    with pytest.raises(b200bgzf.B200BgzfError) as e:
        b200bgzf.index(b"\x1f\x8b\x08\x04" + b"\0" * 40)
    assert e.value.code == b200bgzf.E_FORMAT


def test_offset_and_reindex_usage():
    for args in (["--offset=5"], ["-l6", "--offset=5"], ["-d", "--size=5"], ["--reindex"], ["-d", "--reindex", "--gzi=/dev/null"], ["-d", "--offset=x"]):
        r = subprocess.run([APPLET] + args, input=b"", capture_output=True)
        assert r.returncode == 1 and b"Usage" in r.stderr, args


def test_reindex_writes_the_gzi_of_a_stream(tmp_path):
    for name, _data, stream in list(_emulated_streams()) + list(_golden_streams())[:2]:
        src, gzi = tmp_path / "in.bgz", tmp_path / "out.gzi"
        src.write_bytes(stream)
        with open(src, "rb") as f:
            r = subprocess.run([APPLET, "--reindex", f"--gzi={gzi}"], stdin=f, capture_output=True)
        assert r.returncode == 0 and r.stdout == b"", (name, r.stderr)
        assert gzi.read_bytes() == H.gzi_of(stream), name
        r = subprocess.run([APPLET, "--reindex", f"--gzi={gzi}"], input=stream, capture_output=True)     # (a pipe: read, not mapped)
        assert r.returncode == 0 and gzi.read_bytes() == H.gzi_of(stream), name


def test_offset_past_the_end_is_refused(tmp_path):
    data = H.synth("fastq", 2 * H.BLOCK + 5)
    src = tmp_path / "in.bgz"
    src.write_bytes(H.emul_stream(data, 6))
    with open(src, "rb") as f:
        r = subprocess.run([APPLET, "-d", f"--offset={len(data) + 1}"], stdin=f, capture_output=True)
    assert r.returncode == 1 and b"past the end" in r.stderr and r.stdout == b""


# ---------------------------------------------------------------- GPU


@pytest.fixture(scope="module")
def codec():
    c = b200bgzf.Codec(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def fastq32(codec):
    data = H.synth("fastq", 32 << 20)
    stream, _ = codec.compress_indexed(data, 6)
    return data, stream, b200bgzf.index(stream)


def _device_ranges(codec, stream, ranges, voffsets=False, flags=0):
    import torch
    d_in = torch.frombuffer(bytearray(stream), dtype=torch.uint8).cuda()
    need = ctypes.c_size_t()
    arr = (b200bgzf.Range * max(len(ranges), 1))(*[b200bgzf.Range(b, e) for b, e in ranges])
    fl = flags | (b200bgzf.RANGE_VOFFSET if voffsets else 0)
    rc = codec.lib.b200bgzf_inflate_ranges_device(codec.h, d_in.data_ptr(), len(stream), arr, len(ranges), None, 0, ctypes.byref(need), None, fl, None)
    assert rc in (0, b200bgzf.E_NOSPACE), rc
    d_out = torch.empty(need.value + 64, dtype=torch.uint8, device="cuda")
    n, offs = codec.inflate_ranges_device(d_in.data_ptr(), len(stream), ranges, d_out.data_ptr(), d_out.numel(), voffsets, flags)
    assert n == need.value
    return d_out[:n].cpu().numpy().tobytes(), offs


def _seeded_ranges(total, uaddr, count, max_len, seed):
    rnd = random.Random(seed)
    bounds = [u for u in uaddr if 0 < u < total]
    out = [(0, min(total, 1000)), (total - 500, total), (0, total), (total, total), (0, 0)]
    for k in range(40):                                  # exactly on member boundaries, both ends
        b = rnd.choice(bounds)
        out.append((b, min(total, rnd.choice([u for u in uaddr if u >= b] + [total]))))
        out.append((max(0, b - rnd.randrange(1, 5000)), b))
    while len(out) < count:
        b = rnd.randrange(total + 1)
        out.append((b, min(total, b + rnd.randrange(max_len + 1))))
    rnd.shuffle(out)                                     # unsorted, overlapping
    return out


@gpu
def test_ranges_host_and_device_against_slices(codec, fastq32):
    data, stream, (c, u) = fastq32
    ranges = _seeded_ranges(len(data), u, 2000, 300 << 10, seed=11)
    want, want_off = _slices(data, ranges)
    got, off = codec.inflate_ranges(stream, ranges, index=(c, u))
    assert off == want_off and got == want
    got, off = codec.inflate_ranges(stream, ranges)
    assert off == want_off and got == want
    got, off = _device_ranges(codec, stream, ranges)
    assert off == want_off and got == want
    got, off = codec.inflate_ranges(stream, ranges, index=(c, u), flags=b200bgzf.VERIFY)
    assert got == want


@gpu
def test_ranges_with_a_gzi_index(codec, fastq32):
    data, stream, _ = fastq32
    gc, gu = b200bgzf.gzi_parse(H.gzi_of(stream))        # data members only: the EOF marker is part of the last one's span
    ranges = _seeded_ranges(len(data), gu, 300, 200 << 10, seed=12)
    got, off = codec.inflate_ranges(stream, ranges, index=(gc, gu))
    assert (got, off) == _slices(data, ranges)


def _voff_case(codec, data, level=6):
    stream, moff = codec.compress_indexed(data, level)
    nb = len(moff)
    eof_at = len(stream) - 28
    cstart = moff + [eof_at]
    isz = [min(H.BLOCK, len(data) - b * H.BLOCK) for b in range(nb)]
    rnd = random.Random(3)
    ranges, truth = [], []

    def v(m, uo):
        return (cstart[m] << 16) | uo, (m * H.BLOCK + uo if m < nb else len(data))

    for _ in range(200):
        m0 = rnd.randrange(nb)
        u0 = rnd.choice([0, isz[m0], rnd.randrange(isz[m0] + 1)])
        m1 = rnd.randrange(m0, nb + 1)
        u1 = 0 if m1 == nb else rnd.choice([0, isz[m1], rnd.randrange(isz[m1] + 1)])
        (a, pa), (b, pb) = v(m0, u0), v(m1, u1)
        if pb < pa:
            continue
        ranges.append((a, b))
        truth.append((pa, pb))
    ranges += [(cstart[0] << 16, cstart[1] << 16), (cstart[nb - 1] << 16, eof_at << 16), (0, len(stream) << 16), (eof_at << 16, len(stream) << 16)]
    truth += [(0, isz[0]), ((nb - 1) * H.BLOCK, len(data)), (0, len(data)), (len(data), len(data))]
    return stream, ranges, truth


@gpu
def test_virtual_offsets_on_bam_like_data(codec):
    data = H.bamlike(3 << 20)
    stream, ranges, truth = _voff_case(codec, data)
    want = _slices(data, truth)
    assert codec.inflate_ranges(stream, ranges, voffsets=True) == want
    assert codec.inflate_ranges(stream, ranges, index=b200bgzf.index(stream), voffsets=True) == want
    assert _device_ranges(codec, stream, ranges, voffsets=True) == want


@gpu
def test_golden_reference_streams(codec):
    for name, data, stream in _golden_streams():
        c, u = b200bgzf.index(stream)
        total = len(data)
        ranges = [(0, total), (1, total - 1), (u[1] - 7, u[1] + 9), (u[1], total), (total, total)]
        want = _slices(data, ranges)
        assert codec.inflate_ranges(stream, ranges, flags=b200bgzf.VERIFY) == want, name
        assert _device_ranges(codec, stream, ranges, flags=b200bgzf.VERIFY) == want, name
        vr = [(0, c[1] << 16), (c[1] << 16 | 5, len(stream) << 16), (3, c[1] << 16 | 100)]
        want = _slices(data, [(0, u[1]), (u[1] + 5, total), (3, u[1] + 100)])
        assert codec.inflate_ranges(stream, vr, voffsets=True) == want, name
        assert _device_ranges(codec, stream, vr, voffsets=True) == want, name


@gpu
def test_only_touched_members_are_read(codec):
    data = H.synth("sam", 24 * H.BLOCK + 77)
    stream, _ = codec.compress_indexed(data, 6)
    c, u = b200bgzf.index(stream)
    ranges = [(u[3] + 10, u[5] - 3), (u[12] + 100, u[12] + 200), (u[4], u[4] + 1)]
    want = _slices(data, ranges)
    blob = bytearray(stream)
    m = 8                                                # untouched: its DEFLATE bytes become garbage
    for k in range(c[m] + 18, _cend(c, len(stream), m) - 8):
        blob[k] = (blob[k] * 7 + 91) & 255
    assert _device_ranges(codec, bytes(blob), ranges, flags=b200bgzf.VERIFY) == want
    # host: every byte outside the touched runs [3, 5] and [12] is zero, up to the last run
    for lo, hi in ((0, c[3]), (_cend(c, len(stream), 5), c[12])):
        blob[lo:hi] = bytes(hi - lo)
    blob = bytes(blob)
    assert codec.inflate_ranges(blob, ranges, index=(c, u), flags=b200bgzf.VERIFY) == want
    with pytest.raises(b200bgzf.B200BgzfError):
        codec.inflate(blob, flags=b200bgzf.VERIFY)
    # a touched member's CRC
    crc_at = _cend(c, len(stream), 12) - 8
    bad = bytearray(blob)
    bad[crc_at] ^= 1
    with pytest.raises(b200bgzf.B200BgzfError) as e:
        codec.inflate_ranges(bytes(bad), ranges, index=(c, u), flags=b200bgzf.VERIFY)
    assert e.value.code == b200bgzf.E_CRC
    bad = bytearray(stream)
    bad[crc_at] ^= 1
    with pytest.raises(b200bgzf.B200BgzfError) as e:
        _device_ranges(codec, bytes(bad), ranges, flags=b200bgzf.VERIFY)
    assert e.value.code == b200bgzf.E_CRC


@gpu
def test_errors(codec, fastq32):
    import torch
    data, stream, (c, u) = fastq32
    total = len(data)
    d_in = torch.frombuffer(bytearray(stream), dtype=torch.uint8).cuda()
    d_out = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    cases = [([(10, 5)], False), ([(0, total + 1)], False), ([((c[2] + 1) << 16, c[3] << 16)], True),
             ([(c[2] << 16 | 65281, c[3] << 16)], True), ([(c[3] << 16, c[2] << 16)], True), ([(0, (len(stream) << 16) | 1)], True)]
    for ranges, vo in cases:
        for call in (lambda: codec.inflate_ranges(stream, ranges, voffsets=vo), lambda: codec.inflate_ranges(stream, ranges, index=(c, u), voffsets=vo),
                     lambda: codec.inflate_ranges_device(d_in.data_ptr(), len(stream), ranges, d_out.data_ptr(), d_out.numel(), voffsets=vo)):
            with pytest.raises(b200bgzf.B200BgzfError) as e:
                call()
            assert e.value.code == b200bgzf.E_ARG, ranges
    # a short output buffer: E_NOSPACE with the size needed
    ranges = [(5, 70000), (100, 100), (total - 3000, total)]
    need = 70000 - 5 + 3000
    arr = (b200bgzf.Range * 3)(*[b200bgzf.Range(b, e) for b, e in ranges])
    n = ctypes.c_size_t()
    host_out = bytearray(need)
    rc = codec.lib.b200bgzf_inflate_ranges_host(codec.h, b200bgzf._addr(stream), len(stream), None, None, 0, arr, 3, b200bgzf._addr(host_out), need - 1, ctypes.byref(n), None, 0)
    assert rc == b200bgzf.E_NOSPACE and n.value == need
    rc = codec.lib.b200bgzf_inflate_ranges_device(codec.h, d_in.data_ptr(), len(stream), arr, 3, d_out.data_ptr(), need - 1, ctypes.byref(n), None, 0, None)
    assert rc == b200bgzf.E_NOSPACE and n.value == need


@gpu
def test_applet_offset_size_and_reindex(codec, tmp_path):
    data = H.synth("fastq", 40 * H.BLOCK + 1234)
    raw, bgz, gzi, gzi2 = (tmp_path / n for n in ("in.fq", "in.bgz", "in.gzi", "re.gzi"))
    raw.write_bytes(data)
    with open(raw, "rb") as f, open(bgz, "wb") as o:
        r = subprocess.run([APPLET, "-c", "-l6", f"--gzi={gzi}"], stdin=f, stdout=o, stderr=subprocess.PIPE)
    assert r.returncode == 0, r.stderr
    stream = bgz.read_bytes()
    with open(bgz, "rb") as f:
        r = subprocess.run([APPLET, "--reindex", f"--gzi={gzi2}"], stdin=f, capture_output=True)
    assert r.returncode == 0 and r.stdout == b""
    assert gzi2.read_bytes() == gzi.read_bytes() == H.gzi_of(stream)
    c, u = b200bgzf.gzi_parse(gzi.read_bytes())
    for off, size in ((0, None), (12345, 200000), (u[3], u[5] - u[3]), (len(data) - 10, 1000), (len(data), 5), (777, 0)):
        want = data[off:] if size is None else data[off : off + size]
        for extra in ([], [f"--gzi={gzi}"]):
            args = [APPLET, "-d", f"--offset={off}"] + ([] if size is None else [f"--size={size}"]) + extra
            with open(bgz, "rb") as f:
                r = subprocess.run(args, stdin=f, capture_output=True)
            assert r.returncode == 0 and r.stdout == want, (off, size, extra, r.stderr)
        r = subprocess.run([APPLET, "-d", f"--offset={off}"] + ([] if size is None else [f"--size={size}"]), input=stream, capture_output=True)
        assert r.returncode == 0 and r.stdout == want                                 # from a pipe
    # -d --gzi without --offset: a whole-stream decode as before (the index is not read)
    with open(bgz, "rb") as f:
        r = subprocess.run([APPLET, "-d", "--gzi=/nonexistent"], stdin=f, capture_output=True)
    assert r.returncode == 0 and r.stdout == data


@gpu
def test_256mib_with_10000_ranges_host_equals_device(codec):
    data = H.synth("fastq", 256 << 20, seed=9)
    stream, _ = codec.compress_indexed(data, 6)
    c, u = b200bgzf.index(stream)
    ranges = _seeded_ranges(len(data), u, 10000, 64 << 10, seed=13)
    host, hoff = codec.inflate_ranges(stream, ranges, index=(c, u))
    dev, doff = _device_ranges(codec, stream, ranges)
    assert hoff == doff and host == dev
    assert (host, hoff) == _slices(data, ranges)


_SMALL_BUDGET = r"""
import sys
sys.path[:0] = sys.argv[1:3]
import b200bgzf, helpers as H, test_ranges as T
codec = b200bgzf.Codec(0)
data = H.synth("sam", 6 << 20)
stream, _ = codec.compress_indexed(data, 6)
c, u = b200bgzf.index(stream)
ranges = T._seeded_ranges(len(data), u, 300, 3 << 20, seed=14)
want = T._slices(data, ranges)
assert codec.inflate_ranges(stream, ranges, index=(c, u), flags=b200bgzf.VERIFY) == want
assert codec.inflate_ranges(stream, ranges) == want
assert T._device_ranges(codec, stream, ranges, flags=b200bgzf.VERIFY) == want
print("ok")
"""


@gpu
def test_passes_and_groups_under_a_small_device_budget():
    """1 MiB of scratch: the device variant runs several inflate + gather passes, the host variant many groups and pieces"""
    env = dict(os.environ, B200BGZF_RANGE_BUDGET=str(1 << 20))
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-c", _SMALL_BUDGET, here, os.path.join(H.ROOT, "7bgzf_b200")], capture_output=True, text=True, env=env)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-3000:]
