"""ctypes binding of the C ABI in include/b200bgzf.h — used by tests/ and bench.py only.

The product is the C library (lib7bgzf_b200.so / 7bgzf.so / 7bgzf); this module adds no logic of its own and
never falls back to a CPU path: if the shared library or a GPU is missing the calls raise.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200BGZF_LIB_PATH") or os.path.join(_HERE, "lib7bgzf_b200.so")   # (the checked build: make checked)
HOOK_PATH = os.path.join(_HERE, "7bgzf.so")
APPLET_PATH = os.path.join(_HERE, "7bgzf")

BLOCK_SIZE = 0xFF00
MAX_BLOCK_SIZE = 0x10000
APPEND_EOF = 1
VERIFY = 2
FRAME_MIGZ = 4
RANGE_VOFFSET = 8
E_NOFIT, E_ARG, E_CUDA, E_FORMAT, E_NOSPACE, E_CRC = 1, -1, -2, -3, -4, -5
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")

EXPORTS = [
    "b200bgzf_create", "b200bgzf_destroy", "b200bgzf_strerror", "b200bgzf_last_error", "b200bgzf_compress_bound",
    "b200bgzf_compress_device", "b200bgzf_compress_host", "b200bgzf_compress_blocks_host", "b200bgzf_inflate_size_host",
    "b200bgzf_inflate_device", "b200bgzf_inflate_host", "b200bgzf_profile", "b200bgzf_launch_count", "b200bgzf_parse_method",
    "b200bgzf_host_alloc", "b200bgzf_host_free", "b200bgzf_member_header", "b200bgzf_compress_host_index", "b200bgzf_gzi_format",
    "b200bgzf_multi_create", "b200bgzf_multi_destroy", "b200bgzf_multi_count", "b200bgzf_multi_ctx", "b200bgzf_shard_blocks",
    "b200bgzf_multi_compress_bound", "b200bgzf_multi_compress_host", "b200bgzf_multi_inflate_host",
    "b200bgzf_pieces_gap_bytes", "b200bgzf_compress_pieces_host", "b200bgzf_crc32_combine", "b200bgzf_container_plan",
    "b200bgzf_container_head", "b200bgzf_container_bound", "b200bgzf_container_frame", "b200bgzf_container_compress_host",
    "b200bgzf_inflate_units_host", "b200bgzf_container_units", "b200bgzf_units_free", "b200bgzf_container_inflate_host",
    "b200bgzf_multi_container_bound", "b200bgzf_multi_container_compress_host", "b200bgzf_container_inflate_size",
    "b200bgzf_index_host", "b200bgzf_gzi_parse", "b200bgzf_inflate_ranges_host", "b200bgzf_inflate_ranges_device",
    "b200bgzf_gzip_inflate_device", "b200bgzf_gzip_index_host", "b200bgzf_gzip_index_device", "b200bgzf_gzip_inflate_ranges_host",
    "b200bgzf_gzip_inflate_ranges_device",
]
CONTAINER_GZIP, CONTAINER_MIGZ, CONTAINER_GZINGA, CONTAINER_DICTZIP, CONTAINER_RAZF = 1, 2, 3, 4, 5


class Unit(ctypes.Structure):
    _fields_ = [("in_off", ctypes.c_uint64), ("in_len", ctypes.c_uint32), ("hdr_len", ctypes.c_uint32), ("out_len", ctypes.c_uint32), ("piece", ctypes.c_uint32)]


class PieceSpec(ctypes.Structure):
    _fields_ = [("member_blocks", ctypes.c_uint32), ("head_gap", ctypes.c_uint32), ("tail_gap", ctypes.c_uint32), ("no_final", ctypes.c_uint32),
                ("piece_base", ctypes.c_uint64), ("piece_total", ctypes.c_uint64), ("history", ctypes.c_uint32), ("reserved", ctypes.c_uint32)]


class Range(ctypes.Structure):
    _fields_ = [("beg", ctypes.c_uint64), ("end", ctypes.c_uint64)]


class B200BgzfError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"b200bgzf error {code}: {msg}")
        self.code = code


def load(path=LIB_PATH):
    if not os.path.exists(path):
        raise B200BgzfError(-2, f"{path} is missing: run `make` (there is no CPU fallback)")
    lib = ctypes.CDLL(path)
    vp, sz, u32, i32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_int
    psz = ctypes.POINTER(sz)
    lib.b200bgzf_create.argtypes = [ctypes.POINTER(vp), i32]
    lib.b200bgzf_destroy.argtypes = [vp]
    lib.b200bgzf_destroy.restype = None
    lib.b200bgzf_strerror.argtypes = [i32]
    lib.b200bgzf_strerror.restype = ctypes.c_char_p
    lib.b200bgzf_last_error.argtypes = [vp]
    lib.b200bgzf_last_error.restype = ctypes.c_char_p
    lib.b200bgzf_compress_bound.argtypes = [sz, u32]
    lib.b200bgzf_compress_bound.restype = sz
    lib.b200bgzf_compress_device.argtypes = [vp, vp, sz, u32, i32, vp, sz, psz, ctypes.c_uint, vp]
    lib.b200bgzf_compress_host.argtypes = [vp, vp, sz, u32, i32, vp, sz, psz, ctypes.c_uint]
    lib.b200bgzf_compress_host_index.argtypes = [vp, vp, sz, u32, i32, vp, sz, psz, ctypes.c_uint, ctypes.POINTER(ctypes.c_uint64), sz]
    lib.b200bgzf_gzi_format.argtypes = [ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64), sz, vp, sz]
    lib.b200bgzf_gzi_format.restype = sz
    lib.b200bgzf_compress_blocks_host.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(u32), ctypes.POINTER(vp), psz,
                                                  ctypes.POINTER(i32), u32, i32]
    lib.b200bgzf_inflate_size_host.argtypes = [vp, sz, psz, psz]
    lib.b200bgzf_inflate_device.argtypes = [vp, vp, sz, vp, sz, psz, ctypes.c_uint, vp]
    lib.b200bgzf_inflate_host.argtypes = [vp, vp, sz, vp, sz, psz, ctypes.c_uint]
    lib.b200bgzf_gzip_inflate_device.argtypes = [vp, vp, sz, vp, sz, psz, ctypes.c_uint, vp]
    lib.b200bgzf_profile.argtypes = [vp, i32, ctypes.POINTER(ctypes.c_ulonglong), i32, i32]
    lib.b200bgzf_launch_count.argtypes = [vp]
    lib.b200bgzf_launch_count.restype = ctypes.c_ulonglong
    lib.b200bgzf_parse_method.argtypes = [ctypes.c_char_p, ctypes.POINTER(i32), ctypes.c_char_p, sz]
    lib.b200bgzf_member_header.argtypes = [vp, sz, ctypes.POINTER(ctypes.c_uint64)]
    lib.b200bgzf_member_header.restype = u32
    lib.b200bgzf_multi_create.argtypes = [ctypes.POINTER(vp), ctypes.POINTER(i32), i32]
    lib.b200bgzf_multi_destroy.argtypes = [vp]
    lib.b200bgzf_multi_destroy.restype = None
    lib.b200bgzf_multi_count.argtypes = [vp]
    lib.b200bgzf_multi_ctx.argtypes = [vp, i32]
    lib.b200bgzf_multi_ctx.restype = vp
    lib.b200bgzf_shard_blocks.argtypes = [ctypes.c_uint64, i32, i32, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]
    lib.b200bgzf_shard_blocks.restype = None
    lib.b200bgzf_multi_compress_bound.argtypes = [vp, sz, u32]
    lib.b200bgzf_multi_compress_bound.restype = sz
    lib.b200bgzf_multi_compress_host.argtypes = [vp, vp, sz, u32, i32, vp, sz, psz, ctypes.c_uint]
    lib.b200bgzf_multi_inflate_host.argtypes = [vp, vp, sz, vp, sz, psz, ctypes.c_uint]
    pspec, pu64, pu32 = ctypes.POINTER(PieceSpec), ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(u32)
    lib.b200bgzf_pieces_gap_bytes.argtypes = [sz, u32, pspec]
    lib.b200bgzf_pieces_gap_bytes.restype = sz
    lib.b200bgzf_compress_pieces_host.argtypes = [vp, vp, sz, u32, i32, pspec, vp, sz, psz, pu64, pu32, sz]
    lib.b200bgzf_crc32_combine.argtypes = [u32, u32, ctypes.c_uint64]
    lib.b200bgzf_crc32_combine.restype = u32
    lib.b200bgzf_container_plan.argtypes = [i32, u32, pu32, pspec]
    lib.b200bgzf_container_head.argtypes = [i32, sz]
    lib.b200bgzf_container_head.restype = sz
    lib.b200bgzf_container_bound.argtypes = [i32, u32, sz]
    lib.b200bgzf_container_bound.restype = sz
    lib.b200bgzf_container_frame.argtypes = [i32, u32, vp, sz, sz, pu64, pu32, sz, sz]
    lib.b200bgzf_container_frame.restype = sz
    lib.b200bgzf_container_compress_host.argtypes = [vp, i32, u32, vp, sz, i32, vp, sz, psz]
    punit = ctypes.POINTER(Unit)
    lib.b200bgzf_inflate_units_host.argtypes = [vp, vp, sz, punit, sz, vp, sz, psz, ctypes.c_uint, pu32]
    lib.b200bgzf_container_units.argtypes = [i32, vp, sz, ctypes.POINTER(punit), psz, psz]
    lib.b200bgzf_units_free.argtypes = [punit]
    lib.b200bgzf_units_free.restype = None
    lib.b200bgzf_container_inflate_host.argtypes = [vp, i32, vp, sz, vp, sz, psz, ctypes.c_uint]
    lib.b200bgzf_container_inflate_size.argtypes = [i32, vp, sz, psz, psz]
    lib.b200bgzf_multi_container_bound.argtypes = [vp, i32, u32, sz]
    lib.b200bgzf_multi_container_bound.restype = sz
    lib.b200bgzf_multi_container_compress_host.argtypes = [vp, i32, u32, vp, sz, i32, vp, sz, psz]
    lib.b200bgzf_index_host.argtypes = [vp, sz, pu64, pu64, sz, psz]
    lib.b200bgzf_gzi_parse.argtypes = [vp, sz, pu64, pu64, sz, psz]
    prange = ctypes.POINTER(Range)
    lib.b200bgzf_inflate_ranges_host.argtypes = [vp, vp, sz, pu64, pu64, sz, prange, sz, vp, sz, psz, pu64, ctypes.c_uint]
    lib.b200bgzf_inflate_ranges_device.argtypes = [vp, vp, sz, prange, sz, vp, sz, psz, pu64, ctypes.c_uint, vp]
    lib.b200bgzf_gzip_index_host.argtypes = [vp, vp, sz, u32, vp, sz, psz]
    lib.b200bgzf_gzip_index_device.argtypes = [vp, vp, sz, u32, vp, sz, psz, vp]
    lib.b200bgzf_gzip_inflate_ranges_host.argtypes = [vp, vp, sz, vp, sz, prange, sz, vp, sz, psz, pu64, ctypes.c_uint]
    lib.b200bgzf_gzip_inflate_ranges_device.argtypes = [vp, vp, sz, vp, sz, prange, sz, vp, sz, psz, pu64, ctypes.c_uint, vp]
    return lib


def container_units(kind, blob, lib=None):
    """([(in_off, in_len, hdr_len, out_len, piece)], decoded size) — b200bgzf_container_units; raises on a malformed container"""
    lib = lib or load()
    u, n, total = ctypes.POINTER(Unit)(), ctypes.c_size_t(), ctypes.c_size_t()
    rc = lib.b200bgzf_container_units(kind, _addr(blob), len(blob), ctypes.byref(u), ctypes.byref(n), ctypes.byref(total))
    if rc != 0:
        raise B200BgzfError(rc, "container units")
    try:
        return [(u[i].in_off, u[i].in_len, u[i].hdr_len, u[i].out_len, u[i].piece) for i in range(n.value)], total.value
    finally:
        lib.b200bgzf_units_free(u)


def container_plan(kind, param=0, lib=None):
    """(block size, PieceSpec) of a container — b200bgzf_container_plan"""
    lib = lib or load()
    bs, sp = ctypes.c_uint32(), PieceSpec()
    rc = lib.b200bgzf_container_plan(kind, param, ctypes.byref(bs), ctypes.byref(sp))
    if rc != 0:
        raise B200BgzfError(rc, "container plan")
    return bs.value, sp


def container_frame(kind, param, stream, piece_off, piece_crc, in_bytes, lib=None):
    """b200bgzf_container_frame around a piece stream (bytes): the finished container (one dictzip member)"""
    lib = lib or load()
    n = len(piece_off)
    head = lib.b200bgzf_container_head(kind, n)
    buf = bytearray(head + len(stream) + 64 + 40 * (n + 1))
    buf[head : head + len(stream)] = stream
    off = (ctypes.c_uint64 * max(n, 1))(*piece_off)
    crc = (ctypes.c_uint32 * max(n, 1))(*piece_crc)
    total = lib.b200bgzf_container_frame(kind, param, _addr(buf), len(buf), len(stream), off, crc, n, in_bytes)
    return bytes(buf[:total])


def _addr(buf):
    """address of a bytes / bytearray / ctypes buffer / numpy array / int"""
    if isinstance(buf, int):
        return buf
    if isinstance(buf, bytes):
        return ctypes.cast(ctypes.c_char_p(buf), ctypes.c_void_p).value
    if hasattr(buf, "ctypes"):
        return buf.ctypes.data
    if hasattr(buf, "data_ptr"):
        return buf.data_ptr()
    return ctypes.addressof((ctypes.c_char * len(buf)).from_buffer(buf))


class Codec:
    """One GPU context."""

    def __init__(self, device=-1, path=LIB_PATH):
        self.lib = load(path)
        h = ctypes.c_void_p()
        rc = self.lib.b200bgzf_create(ctypes.byref(h), device)
        if rc != 0:
            raise B200BgzfError(rc, self.lib.b200bgzf_strerror(rc).decode())
        self.h = h

    def close(self):
        if self.h:
            self.lib.b200bgzf_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, ok=(0,)):
        if rc not in ok:
            raise B200BgzfError(rc, self.lib.b200bgzf_strerror(rc).decode() + " / " + self.lib.b200bgzf_last_error(self.h).decode())
        return rc

    def bound(self, n, block_size=BLOCK_SIZE):
        return self.lib.b200bgzf_compress_bound(n, block_size)

    # ---- host buffers ----
    def compress(self, data, level=6, block_size=BLOCK_SIZE, eof=True, flags=0):
        out = bytearray(self.bound(len(data), block_size))
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_compress_host(self.h, _addr(data) if len(data) else None, len(data), block_size, level,
                                                    _addr(out), len(out), ctypes.byref(n), (APPEND_EOF if eof else 0) | flags))
        return bytes(out[: n.value])

    def compress_pieces(self, data, spec, level=6, block_size=BLOCK_SIZE):
        """(piece stream, piece offsets, piece CRCs) — b200bgzf_compress_pieces_host"""
        nb = (len(data) + block_size - 1) // block_size
        cap = self.bound(len(data), block_size) + self.lib.b200bgzf_pieces_gap_bytes(len(data), block_size, ctypes.byref(spec))
        out = bytearray(cap)
        off = (ctypes.c_uint64 * max(nb, 1))()
        crc = (ctypes.c_uint32 * max(nb, 1))()
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_compress_pieces_host(self.h, _addr(data) if len(data) else None, len(data), block_size, level,
                                                           ctypes.byref(spec), _addr(out), len(out), ctypes.byref(n), off, crc, max(nb, 1)))
        return bytes(out[: n.value]), list(off[:nb]), list(crc[:nb])

    def container(self, kind, data, level=6, param=0):
        """a whole container (gzip / MiGz / GZinga / dictzip / RAZF) — b200bgzf_container_compress_host"""
        out = bytearray(self.lib.b200bgzf_container_bound(kind, param, len(data)))
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_container_compress_host(self.h, kind, param, _addr(data) if len(data) else None, len(data), level,
                                                              _addr(out), len(out), ctypes.byref(n)))
        return bytes(out[: n.value])

    def container_inflate(self, kind, blob, flags=0):
        """b200bgzf_container_inflate_host"""
        total = ctypes.c_size_t()
        rc = self.lib.b200bgzf_container_inflate_size(kind, _addr(blob), len(blob), ctypes.byref(total), None)
        if rc != 0:
            raise B200BgzfError(rc, "container size")
        total = total.value
        out = bytearray(max(total, 1))
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_container_inflate_host(self.h, kind, _addr(blob), len(blob), _addr(out), len(out), ctypes.byref(n), flags))
        return bytes(out[: n.value])

    def inflate_units(self, blob, units, out_bytes, flags=0, want_crc=False):
        arr = (Unit * len(units))(*[Unit(*u) for u in units])
        out = bytearray(max(out_bytes, 1))
        n = ctypes.c_size_t()
        crc = (ctypes.c_uint32 * max(len(units), 1))() if want_crc else None
        self._check(self.lib.b200bgzf_inflate_units_host(self.h, _addr(blob), len(blob), arr, len(units), _addr(out), len(out), ctypes.byref(n), flags, crc))
        return (bytes(out[: n.value]), list(crc[: len(units)])) if want_crc else bytes(out[: n.value])

    def compress_indexed(self, data, level=6, block_size=BLOCK_SIZE, eof=True):
        """(stream, member offsets) — b200bgzf_compress_host_index"""
        nb = (len(data) + block_size - 1) // block_size
        out = bytearray(self.bound(len(data), block_size))
        off = (ctypes.c_uint64 * max(nb, 1))()
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_compress_host_index(self.h, _addr(data) if len(data) else None, len(data), block_size, level,
                                                          _addr(out), len(out), ctypes.byref(n), APPEND_EOF if eof else 0, off, nb))
        return bytes(out[: n.value]), list(off[:nb])

    def compress_into(self, src_addr, nbytes, dst_addr, dst_cap, level=6, block_size=BLOCK_SIZE, eof=True):
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_compress_host(self.h, src_addr, nbytes, block_size, level, dst_addr, dst_cap, ctypes.byref(n),
                                                    APPEND_EOF if eof else 0))
        return n.value

    def inflate(self, data, flags=0):
        total, nm = ctypes.c_size_t(), ctypes.c_size_t()
        self._check(self.lib.b200bgzf_inflate_size_host(_addr(data), len(data), ctypes.byref(total), ctypes.byref(nm)))
        out = bytearray(max(total.value, 1))
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_inflate_host(self.h, _addr(data), len(data), _addr(out), len(out), ctypes.byref(n), flags))
        return bytes(out[: n.value])

    def inflate_into(self, src_addr, nbytes, dst_addr, dst_cap, flags=0):
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_inflate_host(self.h, src_addr, nbytes, dst_addr, dst_cap, ctypes.byref(n), flags))
        return n.value

    def compress_blocks(self, payloads, level=6, caps=None):
        nb = len(payloads)
        srcs = (ctypes.c_void_p * nb)(*[_addr(p) if len(p) else None for p in payloads])
        slen = (ctypes.c_uint32 * nb)(*[len(p) for p in payloads])
        bufs = [bytearray(MAX_BLOCK_SIZE) for _ in range(nb)]
        dsts = (ctypes.c_void_p * nb)(*[_addr(b) for b in bufs])
        dlen = (ctypes.c_size_t * nb)(*(caps or [MAX_BLOCK_SIZE] * nb))
        st = (ctypes.c_int * nb)()
        rc = self.lib.b200bgzf_compress_blocks_host(self.h, srcs, slen, dsts, dlen, st, nb, level)
        self._check(rc, ok=(0, 1))
        return [bytes(bufs[i][: dlen[i]]) if st[i] == 0 else None for i in range(nb)], list(st)

    # ---- device buffers (addresses) ----
    def compress_device(self, d_in, nbytes, d_out, out_cap, level=6, block_size=BLOCK_SIZE, eof=True, stream=None):
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_compress_device(self.h, d_in, nbytes, block_size, level, d_out, out_cap, ctypes.byref(n),
                                                      APPEND_EOF if eof else 0, stream))
        return n.value

    def inflate_device(self, d_in, nbytes, d_out, out_cap, flags=0, stream=None):
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_inflate_device(self.h, d_in, nbytes, d_out, out_cap, ctypes.byref(n), flags, stream))
        return n.value

    def gzip_inflate_device(self, d_in, nbytes, d_out, out_cap, flags=0, stream=None):
        """One whole-stream gzip member in device memory -> d_out; returns the decoded size (b200bgzf_gzip_inflate_device)."""
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_gzip_inflate_device(self.h, d_in, nbytes, d_out, out_cap, ctypes.byref(n), flags, stream))
        return n.value

    # ---- random access ----
    def inflate_ranges(self, blob, ranges, index=None, voffsets=False, flags=0):
        """(the ranges' bytes back to back, where each range starts) — b200bgzf_inflate_ranges_host.  ranges: [(beg, end)] of
        the decoded stream, or of BGZF virtual offsets with voffsets=True; index: (caddr, uaddr) as index() / gzi_parse()
        give them, or None (header walk)"""
        n = len(ranges)
        arr = (Range * max(n, 1))(*[Range(b, e) for b, e in ranges])
        ca = ua = None
        ni = 0
        if index is not None:
            ni = len(index[0])
            ca, ua = (ctypes.c_uint64 * max(ni, 1))(*index[0]), (ctypes.c_uint64 * max(ni, 1))(*index[1])
        fl = flags | (RANGE_VOFFSET if voffsets else 0)
        need, off = ctypes.c_size_t(), (ctypes.c_uint64 * max(n, 1))()
        rc = self.lib.b200bgzf_inflate_ranges_host(self.h, _addr(blob), len(blob), ca, ua, ni, arr, n, None, 0, ctypes.byref(need), off, fl)
        self._check(rc, ok=(0, E_NOSPACE))
        out = bytearray(max(need.value, 1))
        got = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_inflate_ranges_host(self.h, _addr(blob), len(blob), ca, ua, ni, arr, n, _addr(out), len(out),
                                                          ctypes.byref(got), off, fl))
        return bytes(out[: got.value]), list(off[:n])

    def inflate_ranges_device(self, d_in, nbytes, ranges, d_out, out_cap, voffsets=False, flags=0, stream=None):
        """(output bytes, where each range starts) — b200bgzf_inflate_ranges_device (device addresses in and out)"""
        n = len(ranges)
        arr = (Range * max(n, 1))(*[Range(b, e) for b, e in ranges])
        got, off = ctypes.c_size_t(), (ctypes.c_uint64 * max(n, 1))()
        self._check(self.lib.b200bgzf_inflate_ranges_device(self.h, d_in, nbytes, arr, n, d_out, out_cap, ctypes.byref(got), off,
                                                            flags | (RANGE_VOFFSET if voffsets else 0), stream))
        return got.value, list(off[:n])

    # ---- whole-stream gzip: random access through a checkpoint index ----
    def _sized(self, fn):
        """fn(buffer, cap, byref(size)) once to learn the size (E_NOSPACE), then into a buffer of that size"""
        need = ctypes.c_size_t()
        self._check(fn(None, 0, ctypes.byref(need)), ok=(0, E_NOSPACE))
        out = bytearray(max(need.value, 1))
        self._check(fn(_addr(out), len(out), ctypes.byref(need)))
        return bytes(out[: need.value])

    def gzip_index(self, blob, span=0):
        """the checkpoint index of one gzip member (bytes) — b200bgzf_gzip_index_host (the member is decoded twice: size, then bytes)"""
        return self._sized(lambda buf, cap, n: self.lib.b200bgzf_gzip_index_host(self.h, _addr(blob), len(blob), span, buf, cap, n))

    def gzip_index_device(self, d_in, nbytes, span=0, stream=None):
        """b200bgzf_gzip_index_device: the index (bytes, host) of the member at device address d_in"""
        return self._sized(lambda buf, cap, n: self.lib.b200bgzf_gzip_index_device(self.h, d_in, nbytes, span, buf, cap, n, stream))

    def gzip_inflate_ranges(self, blob, index, ranges, flags=0):
        """(the ranges' bytes back to back, where each range starts) — b200bgzf_gzip_inflate_ranges_host"""
        n = len(ranges)
        arr = (Range * max(n, 1))(*[Range(b, e) for b, e in ranges])
        need, off = ctypes.c_size_t(), (ctypes.c_uint64 * max(n, 1))()
        self._check(self.lib.b200bgzf_gzip_inflate_ranges_host(self.h, _addr(blob), len(blob), _addr(index), len(index), arr, n, None, 0,
                                                               ctypes.byref(need), off, flags), ok=(0, E_NOSPACE))
        out = bytearray(max(need.value, 1))
        got = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_gzip_inflate_ranges_host(self.h, _addr(blob), len(blob), _addr(index), len(index), arr, n, _addr(out),
                                                               len(out), ctypes.byref(got), off, flags))
        return bytes(out[: got.value]), list(off[:n])

    def gzip_inflate_ranges_device(self, d_in, nbytes, index, ranges, d_out, out_cap, flags=0, stream=None):
        """(output bytes, where each range starts) — b200bgzf_gzip_inflate_ranges_device (device addresses in and out, host index)"""
        n = len(ranges)
        arr = (Range * max(n, 1))(*[Range(b, e) for b, e in ranges])
        got, off = ctypes.c_size_t(), (ctypes.c_uint64 * max(n, 1))()
        self._check(self.lib.b200bgzf_gzip_inflate_ranges_device(self.h, d_in, nbytes, _addr(index), len(index), arr, n, d_out, out_cap,
                                                                 ctypes.byref(got), off, flags, stream))
        return got.value, list(off[:n])

    def profile(self, enable=True, reset=True, slots=32):
        arr = (ctypes.c_ulonglong * slots)()
        self._check(self.lib.b200bgzf_profile(self.h, 1 if enable else 0, arr, slots, 1 if reset else 0))
        return list(arr)

    def launches(self):
        return self.lib.b200bgzf_launch_count(self.h)


class MultiCodec:
    """Several GPU contexts behind one host-buffer call (b200bgzf_multi_*): contiguous block ranges, no collective."""

    def __init__(self, devices, path=LIB_PATH):
        self.lib = load(path)
        h = ctypes.c_void_p()
        arr = (ctypes.c_int * len(devices))(*devices)
        rc = self.lib.b200bgzf_multi_create(ctypes.byref(h), arr, len(devices))
        if rc != 0:
            raise B200BgzfError(rc, self.lib.b200bgzf_strerror(rc).decode())
        self.h = h

    def close(self):
        if self.h:
            self.lib.b200bgzf_multi_destroy(self.h)
            self.h = None

    def count(self):
        return self.lib.b200bgzf_multi_count(self.h)

    def bound(self, n, block_size=BLOCK_SIZE):
        return self.lib.b200bgzf_multi_compress_bound(self.h, n, block_size)

    def _check(self, rc):
        if rc != 0:
            raise B200BgzfError(rc, self.lib.b200bgzf_strerror(rc).decode())

    def compress_into(self, src_addr, nbytes, dst_addr, dst_cap, level=6, block_size=BLOCK_SIZE, eof=True, flags=0):
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_multi_compress_host(self.h, src_addr, nbytes, block_size, level, dst_addr, dst_cap, ctypes.byref(n),
                                                          (APPEND_EOF if eof else 0) | flags))
        return n.value

    def compress(self, data, level=6, block_size=BLOCK_SIZE, eof=True, flags=0):
        out = bytearray(self.bound(len(data), block_size))
        n = self.compress_into(_addr(data) if len(data) else None, len(data), _addr(out), len(out), level, block_size, eof, flags)
        return bytes(out[:n])

    def container(self, kind, data, level=6, param=0):
        """b200bgzf_multi_container_compress_host"""
        out = bytearray(self.lib.b200bgzf_multi_container_bound(self.h, kind, param, len(data)))
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_multi_container_compress_host(self.h, kind, param, _addr(data) if len(data) else None, len(data), level,
                                                                    _addr(out), len(out), ctypes.byref(n)))
        return bytes(out[: n.value])

    def inflate_into(self, src_addr, nbytes, dst_addr, dst_cap, flags=0):
        n = ctypes.c_size_t()
        self._check(self.lib.b200bgzf_multi_inflate_host(self.h, src_addr, nbytes, dst_addr, dst_cap, ctypes.byref(n), flags))
        return n.value

    def inflate(self, data, flags=0):
        total, nm = ctypes.c_size_t(), ctypes.c_size_t()
        self._check(self.lib.b200bgzf_inflate_size_host(_addr(data), len(data), ctypes.byref(total), ctypes.byref(nm)))
        out = bytearray(max(total.value, 1))
        n = self.inflate_into(_addr(data), len(data), _addr(out), len(out), flags)
        return bytes(out[:n])


def shard_blocks(nblocks, shard, nshards, lib=None):
    lib = lib or load()
    a, b = ctypes.c_uint64(), ctypes.c_uint64()
    lib.b200bgzf_shard_blocks(nblocks, shard, nshards, ctypes.byref(a), ctypes.byref(b))
    return a.value, b.value


def member_header(data, lib=None):
    """(header length, member size) of the gzip member at the front of `data` (any flavour of applet/7bgzf.c:81-131), or (0, 0)"""
    lib = lib or load()
    n = ctypes.c_uint64()
    h = lib.b200bgzf_member_header(_addr(data), len(data), ctypes.byref(n))
    return h, n.value


def gzi_format(caddr, uaddr, lib=None):
    """bytes of the .gzi for members starting at (caddr[i], uaddr[i]) — b200bgzf_gzi_format"""
    lib = lib or load()
    n = len(caddr)
    ca, ua = (ctypes.c_uint64 * max(n, 1))(*caddr), (ctypes.c_uint64 * max(n, 1))(*uaddr)
    buf = bytearray(8 + 16 * max(n - 1, 0))
    w = lib.b200bgzf_gzi_format(ca, ua, n, _addr(buf), len(buf))
    return bytes(buf[:w])


def _pairs(fn, blob, what, lib):
    n = ctypes.c_size_t()
    rc = fn(_addr(blob), len(blob), None, None, 0, ctypes.byref(n))
    if rc not in (0, E_NOSPACE):
        raise B200BgzfError(rc, what)
    ca, ua = (ctypes.c_uint64 * max(n.value, 1))(), (ctypes.c_uint64 * max(n.value, 1))()
    rc = fn(_addr(blob), len(blob), ca, ua, n.value, ctypes.byref(n))
    if rc != 0:
        raise B200BgzfError(rc, what)
    return list(ca[: n.value]), list(ua[: n.value])


def index(blob, lib=None):
    """(caddr, uaddr): start of every member (EOF marker included) in the stream and in its decoded bytes — b200bgzf_index_host"""
    lib = lib or load()
    return _pairs(lib.b200bgzf_index_host, blob, "member index", lib)


def gzi_parse(data, lib=None):
    """(caddr, uaddr) of a .gzi, the implicit (0, 0) entry first — b200bgzf_gzi_parse"""
    lib = lib or load()
    return _pairs(lib.b200bgzf_gzi_parse, data, ".gzi", lib)
