"""ctypes access to the TEST infrastructure: synthetic data, the CPU thread-emulator of the block encoder,
the oracle restatement (oracle/liboracle.so) and the compiled reference (oracle/_ref/7bgzf_ref.so)."""
import ctypes
import functools
import gzip
import os
import struct
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "7bgzf_ref.so")
REF_7BGZF = os.path.join(ROOT, "oracle", "_ref", "7bgzf")
GOLDEN = os.path.join(ROOT, "tests", "golden")
BLOCK = 0xFF00
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")

vp, sz, u8p = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_char_p


@functools.lru_cache(None)
def _gen():
    lib = ctypes.CDLL(os.path.join(ROOT, "build", "libdatagen.so"))
    lib.b200gen_fill.argtypes = [ctypes.c_int, ctypes.c_uint64, vp, sz]
    lib.b200gen_fill.restype = sz
    return lib


def synth(kind, nbytes, seed=None):
    """kind: 'fastq' | 'sam' — SURVEY.md Appendix B generator (seed 1 / 2 by default)"""
    k = 0 if kind == "fastq" else 1
    buf = ctypes.create_string_buffer(nbytes)
    _gen().b200gen_fill(k, seed if seed is not None else 1 + k, buf, nbytes)
    return buf.raw


def lcg_noise(n):
    x, out = 12345, bytearray()
    for _ in range(n):
        x = (x * 1664525 + 1013904223) & 0xFFFFFFFF
        out.append(x >> 24)
    return bytes(out)


def acgt(n):
    return bytes(b"ACGT"[(i * 7 + i // 3) & 3] for i in range(n))


@functools.lru_cache(None)
def _emul():
    lib = ctypes.CDLL(os.path.join(ROOT, "build", "libemul.so"))
    lib.bgemul_compress_block.argtypes = [u8p, ctypes.c_uint32, ctypes.c_int, ctypes.c_int, u8p, ctypes.POINTER(ctypes.c_uint32)]
    lib.bgemul_set_header_bytes.argtypes = [ctypes.c_uint32]
    lib.bgemul_set_header_bytes.restype = None
    return lib


def emul_block(payload, level=6, order=0):
    dst = ctypes.create_string_buffer(65536)
    dl = ctypes.c_uint32()
    rc = _emul().bgemul_compress_block(payload, len(payload), level, order, dst, ctypes.byref(dl))
    return rc, dst.raw[: dl.value]


def emul_trees():
    """the trees of the last emulated block's final pass: {btype, (used symbols, overflow) of "litlen", "dist", "precode"};
    overflow = nodes deeper than the code's length limit (15, 15, 7), what the code-length repair starts from"""
    lib = _emul()
    lib.bgemul_last_trees.argtypes = [ctypes.POINTER(ctypes.c_uint32)]
    lib.bgemul_last_trees.restype = None
    v = (ctypes.c_uint32 * 7)()
    lib.bgemul_last_trees(v)
    return {"btype": v[0], "litlen": (v[1], v[2]), "dist": (v[3], v[4]), "precode": (v[5], v[6])}


def emul_ties():
    """ties in the last emulated block's distance and precode trees: {"dist" / "precode": (leaves of the same weight as
    the leaf before them, merge picks where the lightest leaf and the lightest merged node weigh the same)}"""
    lib = _emul()
    lib.bgemul_last_ties.argtypes = [ctypes.POINTER(ctypes.c_uint32)]
    lib.bgemul_last_ties.restype = None
    v = (ctypes.c_uint32 * 4)()
    lib.bgemul_last_ties(v)
    return {"dist": (v[0], v[1]), "precode": (v[2], v[3])}


def emul_piece(payload, level=6, head_gap=0, tail_gap=0, final=True, order=0, history=b""):
    """One block in piece mode (raw DEFLATE between `head_gap` and `tail_gap` free bytes): (slot bytes, CRC-32 of payload).
    history: the input right before the payload that matches may reach into (a multiple of 272 bytes, at most 32640)."""
    lib = _emul()
    lib.bgemul_set_piece.argtypes = [ctypes.c_uint32] * 4
    lib.bgemul_set_piece.restype = None
    lib.bgemul_set_history.argtypes = [ctypes.c_uint32]
    lib.bgemul_set_history.restype = None
    lib.bgemul_last_crc.restype = ctypes.c_uint32
    lib.bgemul_set_piece(1, head_gap, tail_gap, 1 if final else 0)
    lib.bgemul_set_history(len(history))
    try:
        rc, m = emul_block(history + payload, level, order)
        if rc == 1:
            raise OverflowError("the piece does not fit its slot")
        assert rc == 0, rc
        return m, lib.bgemul_last_crc()
    finally:
        lib.bgemul_set_piece(0, 0, 0, 1)
        lib.bgemul_set_history(0)


def emul_stream(data, level=6, block=BLOCK, order=0, eof=True):
    out = bytearray()
    for off in range(0, len(data), block):
        rc, m = emul_block(data[off : off + block], level, order)
        assert rc == 0, rc
        out += m
    return bytes(out) + (EOF_BLOCK if eof else b"")


@functools.lru_cache(None)
def oracle():
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "liboracle.so"))
    lib.oracle_crc32.argtypes = [ctypes.c_uint32, u8p, sz]
    lib.oracle_crc32.restype = ctypes.c_uint32
    lib.oracle_crc32_combine.argtypes = [ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint64]
    lib.oracle_crc32_combine.restype = ctypes.c_uint32
    lib.oracle_eof_block.argtypes = [u8p]
    lib.oracle_eof_block.restype = sz
    lib.oracle_bgzf_frame.argtypes = [u8p, u8p, sz, u8p, sz]
    lib.oracle_bgzf_frame.restype = sz
    lib.oracle_store_deflate.argtypes = [u8p, ctypes.POINTER(sz), u8p, sz]
    lib.oracle_read_gz_header.argtypes = [u8p, ctypes.c_int] + [ctypes.POINTER(ctypes.c_int)] * 3
    lib.oracle_inflate.argtypes = [u8p, ctypes.POINTER(sz), u8p, sz]
    lib.oracle_bgzf_decompress.argtypes = [u8p, sz, u8p, sz, ctypes.POINTER(sz), ctypes.POINTER(sz)]
    lib.oracle_parse_method.argtypes = [u8p, ctypes.POINTER(ctypes.c_int)]
    lib.oracle_passthrough.argtypes = [ctypes.c_int]
    # reference harness
    lib.refh_open.argtypes = [u8p, ctypes.c_int]
    lib.refh_open.restype = vp
    lib.refh_close.argtypes = [vp]
    lib.refh_bgzf_compress.argtypes = [vp, u8p, ctypes.POINTER(sz), u8p, sz]
    lib.refh_crc32.argtypes = [vp, u8p, sz]
    lib.refh_crc32.restype = ctypes.c_uint32
    lib.refh_compress.argtypes = [vp, vp, sz, sz, ctypes.c_int, vp, vp, ctypes.POINTER(ctypes.c_int)]
    lib.refh_compress.restype = ctypes.c_double
    lib.refh_inflate.argtypes = [vp, vp, sz, ctypes.c_int, vp, sz, ctypes.POINTER(sz), ctypes.POINTER(ctypes.c_int)]
    lib.refh_inflate.restype = ctypes.c_double
    return lib


def oracle_inflate_raw(deflated, cap):
    out = ctypes.create_string_buffer(max(cap, 1))
    n = sz(cap)
    rc = oracle().oracle_inflate(out, ctypes.byref(n), deflated, len(deflated))
    return rc, out.raw[: n.value]


def oracle_decompress(stream):
    cap = sum(m[2] for m in members(stream)) if stream else 0
    out = ctypes.create_string_buffer(max(cap, 1))
    n, nm = sz(), sz()
    rc = oracle().oracle_bgzf_decompress(stream, len(stream), out, cap, ctypes.byref(n), ctypes.byref(nm))
    return rc, out.raw[: n.value], nm.value


def members(stream):
    """[(offset, size, isize, crc)] by walking BSIZE"""
    out, off = [], 0
    while off < len(stream):
        assert stream[off : off + 4] == b"\x1f\x8b\x08\x04", f"bad magic at {off}"
        size = struct.unpack_from("<H", stream, off + 16)[0] + 1
        crc, isize = struct.unpack_from("<II", stream, off + size - 8)
        out.append((off, size, isize, crc))
        off += size
    assert off == len(stream)
    return out


def gzi_of(stream):
    """the .gzi htslib writes next to a stream it compressed itself: u64 count, then (compressed, uncompressed) offset of
    every member that carries data except the first — from a header walk (oracle for b200bgzf_gzi_format / --gzi)"""
    pairs, u = [], 0
    for off, _size, isize, _crc in members(stream):
        if isize:
            pairs.append((off, u))
        u += isize
    body = b"".join(struct.pack("<QQ", c, a) for c, a in pairs[1:])
    return struct.pack("<Q", max(len(pairs) - 1, 0)) + body


def have_ref():
    return os.path.exists(REF_SO)


class Ref:
    """the unmodified reference (oracle/_ref) at one libdeflate level"""

    _cache = {}

    def __new__(cls, level=6):
        if level not in cls._cache:
            self = super().__new__(cls)
            self.level = level
            self.h = oracle().refh_open(REF_SO.encode(), level)
            assert self.h, "cannot open oracle/_ref/7bgzf_ref.so"
            cls._cache[level] = self
        return cls._cache[level]

    def bgzf_compress(self, payload, cap=65536):
        dst = ctypes.create_string_buffer(max(cap, 1))
        dl = sz(cap)
        rc = oracle().refh_bgzf_compress(self.h, dst, ctypes.byref(dl), payload, len(payload))
        return rc, dst.raw[: dl.value] if rc == 0 else b"", dl.value

    def crc32(self, data):
        return oracle().refh_crc32(self.h, data, len(data))

    def compress_stream(self, data, block=BLOCK, threads=1, keep=True):
        nb = (len(data) + block - 1) // block
        sizes = (ctypes.c_uint32 * max(nb, 1))()
        slots = ctypes.create_string_buffer(max(nb, 1) * 65536) if keep else None
        rc = ctypes.c_int()
        src = ctypes.create_string_buffer(data, len(data)) if not isinstance(data, ctypes.Array) else data
        t = oracle().refh_compress(self.h, ctypes.addressof(src), len(data), block, threads, ctypes.addressof(slots) if keep else None,
                                   ctypes.addressof(sizes), ctypes.byref(rc))
        assert rc.value == 0
        if not keep:
            return None, list(sizes)[:nb], t
        base = ctypes.addressof(slots)
        out = b"".join(ctypes.string_at(base + b * 65536, sizes[b]) for b in range(nb))
        return out, list(sizes)[:nb], t

    def inflate_stream(self, stream, threads=1):
        cap = sum(m[2] for m in members(stream))
        out = ctypes.create_string_buffer(max(cap, 1))
        n, rc = sz(), ctypes.c_int()
        src = ctypes.create_string_buffer(stream, len(stream))
        t = oracle().refh_inflate(self.h, ctypes.addressof(src), len(stream), threads, ctypes.addressof(out), cap, ctypes.byref(n), ctypes.byref(rc))
        return rc.value if t >= 0 else -1, out.raw[: n.value], t


def zlib_member(payload, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    """a BGZF member made by zlib (what htslib without libdeflate writes)"""
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    raw = co.compress(payload) + co.flush()
    return (bytes.fromhex("1f8b08040000000000ff060042430200") + struct.pack("<H", len(raw) + 25) + raw +
            struct.pack("<II", zlib.crc32(payload), len(payload)))


def gunzip(stream):
    return gzip.decompress(stream)


def bamlike(n, seed=5):
    """A BAM-shaped binary record stream made from the SAM-like text (what htslib hands to bgzf_compress when samtools
    writes BAM, BASELINE config 5): 32-byte little-endian core, NUL-terminated name, one CIGAR word, 4-bit packed bases,
    raw Phred bytes, a few binary tags.  Not a valid BAM file; it has BAM's byte statistics."""
    import random, struct
    rnd = random.Random(seed)
    out = bytearray()
    code = {65: 1, 67: 2, 71: 4, 84: 8, 78: 15}
    for l in synth("sam", 2 * n).split(b"\n"):
        f = l.split(b"\t")
        if l.startswith(b"@") or len(f) < 11:
            continue
        seq, qual, name = f[9], f[10], f[0] + b"\0"
        packed = bytes(((code.get(seq[i], 15) << 4) | (code.get(seq[i + 1], 15) if i + 1 < len(seq) else 0)) for i in range(0, len(seq), 2))
        core = struct.pack("<iiBBHHHIiii", 0, int(f[3]) & 0x7fffffff, len(name) & 255, int(f[4]) & 255, 4681, 1, int(f[1]) & 0xffff, len(seq), 0,
                           int(f[7]) & 0x7fffffff, max(-2**31, min(2**31 - 1, int(f[8]))))
        tags = b"NMC" + bytes([rnd.randrange(4)]) + b"ASC" + bytes([150 - rnd.randrange(10)]) + b"RGZgrp1\0"
        rec = core + name + struct.pack("<I", len(seq) << 4) + packed + bytes(max(0, c - 33) for c in qual) + tags
        out += struct.pack("<I", len(rec)) + rec
        if len(out) >= n:
            break
    return bytes(out[:n])


# ---- the other containers (SURVEY 8f ranks 3, 4): pieces from the emulator + the library's framing (no GPU) ----
REF_CIELBOX = os.path.join(ROOT, "oracle", "_ref", "cielbox_ref")
DICTZIP_MAX_CHUNKS = 32762


def codec_module():
    import sys
    sys.path.insert(0, os.path.join(ROOT, "7bgzf_b200"))
    import b200bgzf
    return b200bgzf


def emul_container(kind, data, level=6, param=0):
    """The container b200bgzf_container_compress_host writes, with the emulator standing in for the kernel."""
    B = codec_module()
    lib = B.load()
    bs, sp = B.container_plan(kind, param, lib)
    if kind == B.CONTAINER_MIGZ and not param & 0x80000000:
        try:
            return _emul_container(B, lib, kind, data, level, param)
        except OverflowError:                      # a 64 KiB piece that does not compress: the library redoes the file with small pieces
            return _emul_container(B, lib, kind, data, level, param | 0x80000000)
    return _emul_container(B, lib, kind, data, level, param)


def _emul_container(B, lib, kind, data, level, param):
    bs, sp = B.container_plan(kind, param, lib)
    blocks = [data[i : i + bs] for i in range(0, len(data), bs)]
    per = DICTZIP_MAX_CHUNKS if kind == B.CONTAINER_DICTZIP else max(len(blocks), 1)
    out, done = bytearray(), 0
    while True:
        part = blocks[done : done + per]
        stream, offs, crcs = bytearray(), [], []
        for i, b in enumerate(part):
            first = i % sp.member_blocks == 0
            last = (i + 1) % sp.member_blocks == 0 or i + 1 == len(part)
            # dictionary priming: what precedes the piece inside its member, as far as the window reaches (multiples of 272)
            o = (done + i) * bs
            h = min(sp.history, (i % sp.member_blocks) * bs)
            h -= h % 272
            m, crc = emul_piece(b, level, sp.head_gap if first else 0, sp.tail_gap if last else 0, last and not sp.no_final, history=data[o - h : o])
            offs.append(len(stream))
            crcs.append(crc)
            stream += m
        out += B.container_frame(kind, param, bytes(stream), offs, crcs, sum(map(len, part)), lib)
        done += len(part)
        if done >= len(blocks):
            return bytes(out)


def ref_applet_decode(applet, blob):
    """Decode `blob` with the reference's own applet (7gzip / 7migz read stdin; 7gzinga / 7dictzip / 7razf take a file)."""
    import subprocess, tempfile
    with tempfile.NamedTemporaryFile(delete=False) as f:
        f.write(blob)
        name = f.name
    try:
        if applet in ("7gzip", "7migz", "7bgzf"):
            with open(name, "rb") as fin:
                r = subprocess.run([REF_CIELBOX, applet, "-d"], stdin=fin, capture_output=True)
        else:
            r = subprocess.run([REF_CIELBOX, applet, "-cd", name], capture_output=True)
        return r.returncode, r.stdout
    finally:
        os.unlink(name)
