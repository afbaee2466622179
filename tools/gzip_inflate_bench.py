"""Whole-stream gzip read on one GPU: b200bgzf_gzip_inflate_device and b200bgzf_container_inflate_host(GZIP) against the
one-warp path and, as the yardstick, b200bgzf_inflate_device of the same data as BGZF level 6.

  python tools/gzip_inflate_bench.py [--gib 1] [--reps 10] [--out FILE]

Inputs (FASTQ-like, generator seed 1): (a) our GZIP container at level 6, primed 48 KiB pieces (a flush point every piece);
(b) a pigz-like zlib level-6 stream: 128 KiB chunks primed with the 32 KiB before them, a sync flush after each (built on the
host cores, as pigz builds it); (c) the worst case: 30 KiB of noise repeated to 64 MiB, a sync flush every 40 KiB (every chunk
depends on the one before it).  Per input: device-resident call time (median of `reps` after a warm-up, with min / max; the
call synchronises, the host clock is read around it; inputs are larger than L2), end-to-end container_inflate_host from and to
pinned host buffers, `7gzip -d` wall time (stdin a file, stdout /dev/null), and the one-warp path on a 32 MiB slice.  The
card's name and power limit are read in the same run.
"""
import argparse
import ctypes
import os
import statistics
import struct
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ProcessPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "7bgzf_b200"), os.path.join(ROOT, "tests")]
import b200bgzf as B  # noqa: E402
import helpers as H  # noqa: E402

CHUNK = 128 << 10


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return f"nvidia-smi unavailable ({e})"


_DATA = None


def _init(path):
    global _DATA
    _DATA = open(path, "rb").read()


def _chunk(i):
    beg, end = i * CHUNK, min(len(_DATA), (i + 1) * CHUNK)
    z = zlib.compressobj(6, zlib.DEFLATED, -15, zdict=_DATA[max(0, beg - 32768) : beg]) if beg else zlib.compressobj(6, zlib.DEFLATED, -15)
    return z.compress(_DATA[beg:end]) + z.flush(zlib.Z_FINISH if end == len(_DATA) else zlib.Z_SYNC_FLUSH)


def pigz_like(data):
    with tempfile.NamedTemporaryFile() as f:
        f.write(data)
        f.flush()
        n = (len(data) + CHUNK - 1) // CHUNK
        with ProcessPoolExecutor(os.cpu_count(), initializer=_init, initargs=(f.name,)) as ex:
            body = b"".join(ex.map(_chunk, range(n), chunksize=64))
    return b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\x03" + body + struct.pack("<II", zlib.crc32(data), len(data) & 0xFFFFFFFF)


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), min(ts), max(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say(f"card: {card()}")
    nbytes = int(args.gib * (1 << 30))
    codec = B.Codec(0)
    data = H.synth("fastq", nbytes)
    lib, h = codec.lib, codec.h

    def rate(n, t):
        return n / t / 1e9

    # yardstick: the same data as BGZF level 6 through inflate_device
    bgzf = codec.compress(data, 6)
    d_b = torch.frombuffer(bytearray(bgzf), dtype=torch.uint8).cuda()
    d_out = torch.empty(nbytes + 64, dtype=torch.uint8, device="cuda")
    med, lo, hi = timed(lambda: codec.inflate_device(d_b.data_ptr(), len(bgzf), d_out.data_ptr(), nbytes), args.reps)
    yard = rate(nbytes, med)
    say(f"BGZF L6 inflate_device ({len(bgzf)} B): median {med * 1e3:.1f} ms ({yard:.1f} GB/s), min {lo * 1e3:.1f}, max {hi * 1e3:.1f}")
    del d_b

    t0 = time.perf_counter()
    pig = pigz_like(data)
    say(f"(pigz-like stream built on {os.cpu_count()} host cores in {time.perf_counter() - t0:.1f} s)")
    inputs = [("7gzip primed L6", codec.container(B.CONTAINER_GZIP, data, 6), data),
              ("zlib L6, sync flush / 128 KiB", pig, data)]
    noise = (H.lcg_noise(30 << 10) * ((64 << 20) // (30 << 10) + 1))[: 64 << 20]
    z = zlib.compressobj(6, zlib.DEFLATED, 31)
    worst = b"".join(z.compress(noise[i : i + (40 << 10)]) + z.flush(zlib.Z_SYNC_FLUSH) for i in range(0, len(noise), 40 << 10)) + z.flush()
    inputs.append(("worst case: 30 KiB noise x N, sync flush / 40 KiB, 64 MiB", worst, noise))

    lib.b200bgzf_host_alloc.restype = ctypes.c_void_p
    for name, blob, want in inputs:
        n = len(want)
        say(f"--- {name}: {len(blob)} B -> {n} B")
        d_in = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
        got = codec.gzip_inflate_device(d_in.data_ptr(), len(blob), d_out.data_ptr(), nbytes + 64)
        ok = got == n and zlib.crc32(d_out[:n].cpu().numpy().tobytes()) == zlib.crc32(want)
        med, lo, hi = timed(lambda: codec.gzip_inflate_device(d_in.data_ptr(), len(blob), d_out.data_ptr(), nbytes + 64), args.reps)
        say(f"  gzip_inflate_device: median {med * 1e3:.1f} ms ({rate(n, med):.2f} GB/s = {rate(n, med) / yard:.2f} x BGZF, "
            f"{rate(n, med) / 0.46:.0f} x 0.46 GB/s), min {lo * 1e3:.1f}, max {hi * 1e3:.1f}; output {'correct' if ok else 'WRONG'}")
        del d_in
        p_in = lib.b200bgzf_host_alloc(len(blob))
        p_out = lib.b200bgzf_host_alloc(n + 64)
        ctypes.memmove(p_in, blob, len(blob))
        cnt = ctypes.c_size_t()

        def host():
            rc = lib.b200bgzf_container_inflate_host(h, B.CONTAINER_GZIP, p_in, len(blob), p_out, n + 64, ctypes.byref(cnt), 0)
            assert rc == 0, rc

        med, lo, hi = timed(host, max(3, args.reps // 2))
        ok = zlib.crc32(ctypes.string_at(p_out, n)) == zlib.crc32(want)
        say(f"  container_inflate_host (pinned): median {med * 1e3:.1f} ms ({rate(n, med):.2f} GB/s), min {lo * 1e3:.1f}, "
            f"max {hi * 1e3:.1f}; output {'correct' if ok else 'WRONG'}")
        lib.b200bgzf_host_free(ctypes.c_void_p(p_in))
        lib.b200bgzf_host_free(ctypes.c_void_p(p_out))
        with tempfile.NamedTemporaryFile() as f:
            f.write(blob)
            f.flush()
            exe = os.path.join(ROOT, "7bgzf_b200", "7gzip")
            t0 = time.perf_counter()
            with open(f.name, "rb") as fi, open(os.devnull, "wb") as fo:
                r = subprocess.run([exe, "-d"], stdin=fi, stdout=fo, stderr=subprocess.PIPE)
            t = time.perf_counter() - t0
            say(f"  7gzip -d: {t:.2f} s wall ({rate(n, t):.2f} GB/s), exit {r.returncode}, stderr {r.stderr.decode().strip()!r}")

    # the one-warp path on a 32 MiB slice (our primed file)
    sl = codec.container(B.CONTAINER_GZIP, data[: 32 << 20], 6)
    units, total = B.container_units(B.CONTAINER_GZIP, sl)
    t0 = time.perf_counter()
    out = codec.inflate_units(sl, units, total)
    t = time.perf_counter() - t0
    say(f"one warp (inflate_units, 32 MiB primed 7gzip slice): {t:.2f} s ({rate(32 << 20, t) * 1e3:.1f} MB/s); "
        f"output {'correct' if out == data[: 32 << 20] else 'WRONG'}")
    codec.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
