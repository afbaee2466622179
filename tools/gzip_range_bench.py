"""Random access into a whole-stream gzip member on one GPU: b200bgzf_gzip_index_device and
b200bgzf_gzip_inflate_ranges_device against b200bgzf_gzip_inflate_device of the same file, and a single-core zlib baseline.

  python tools/gzip_range_bench.py [--gib 1] [--reps 10] [--out FILE]

Input: FASTQ-like data (generator seed 1), our GZIP container at level 6 (primed 48 KiB pieces), resident on the device;
index span 1 MiB.  Every GPU number is the median of `reps` calls after 2 warm-ups, with min / max; every call synchronises
and the host clock is read around it; the file is larger than L2.  Reported: index build against gzip_inflate_device;
(a) 1000 random 4 KiB ranges, (b) 1000 random 1 MiB ranges, (c) one 512 MiB range, each as call time, ranges/s, output GB/s
and touched chunks; the index size; zlib on one host core restarting at the same access points with the stored windows
(a sample of the ranges of (a), timed range by range).  The card's name and power limit are read in the same run.
"""
import argparse
import ctypes
import os
import random
import statistics
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "7bgzf_b200"), os.path.join(ROOT, "tests")]
import b200bgzf as B  # noqa: E402
import helpers as H  # noqa: E402
import test_gzip_ranges as G  # noqa: E402

MIB = 1 << 20


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return f"nvidia-smi unavailable ({e})"


def timed(fn, reps):
    fn()
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), min(ts), max(ts)


def plan(x, ranges):
    """per range: (access point chunk, last chunk); and the number of chunks the merged runs touch"""
    us = [u for _, u, _ in x["chunks"]]
    pts = [c for c, _ in x["points"]]
    import bisect
    runs = []
    for b, e in ranges:
        if b == e:
            continue
        f = bisect.bisect_right(us, b) - 1
        last = bisect.bisect_right(us, e - 1) - 1
        runs.append((pts[bisect.bisect_right(pts, f) - 1], last))
    runs.sort()
    touched, cur = 0, None
    for s, e in runs:
        if cur and s <= cur[1] + 1:
            cur[1] = max(cur[1], e)
        else:
            if cur:
                touched += cur[1] - cur[0] + 1
            cur = [s, e]
    if cur:
        touched += cur[1] - cur[0] + 1
    return runs, touched


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--sample", type=int, default=50)
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
    lib, h = codec.lib, codec.h
    data = H.synth("fastq", nbytes)
    blob = codec.container(B.CONTAINER_GZIP, data, 6)
    say(f"input: FASTQ-like {nbytes} B, 7gzip primed L6 -> {len(blob)} B, device-resident; span 1 MiB")
    d_in = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
    d_out = torch.empty(nbytes + 64, dtype=torch.uint8, device="cuda")

    med, lo, hi = timed(lambda: codec.gzip_inflate_device(d_in.data_ptr(), len(blob), d_out.data_ptr(), nbytes + 64), args.reps)
    whole = nbytes / med / 1e9
    say(f"gzip_inflate_device: median {med * 1e3:.1f} ms ({whole:.2f} GB/s), min {lo * 1e3:.1f}, max {hi * 1e3:.1f}")
    cap = 64 * MIB + nbytes // 16
    buf = ctypes.create_string_buffer(cap)
    n = ctypes.c_size_t()

    def build():
        rc = lib.b200bgzf_gzip_index_device(h, d_in.data_ptr(), len(blob), 0, buf, cap, ctypes.byref(n), None)
        assert rc == 0, rc

    imed, ilo, ihi = timed(build, args.reps)
    ix = buf.raw[: n.value]
    assert ix == codec.gzip_index(blob)
    x = G.parse_index(ix)
    say(f"index build (gzip_index_device): median {imed * 1e3:.1f} ms = {imed / med:.2f} x gzip_inflate_device (target <= 1.15), "
        f"min {ilo * 1e3:.1f}, max {ihi * 1e3:.1f}")
    say(f"index: {len(ix)} B ({len(ix) / len(blob) * 100:.2f} % of the file): {len(x['chunks'])} chunks, {len(x['points'])} access points")

    rnd = random.Random(1)
    cases = [("(a) 1000 random 4 KiB ranges", [(b, b + 4096) for b in (rnd.randrange(nbytes - 4096) for _ in range(1000))]),
             ("(b) 1000 random 1 MiB ranges", [(b, b + MIB) for b in (rnd.randrange(nbytes - MIB) for _ in range(1000))])]
    b0 = rnd.randrange(nbytes - 512 * MIB)
    cases.append(("(c) one 512 MiB range", [(b0, b0 + 512 * MIB)]))
    rate_a = None
    for name, rs in cases:
        total = sum(e - b for b, e in rs)
        got, off = codec.gzip_inflate_ranges_device(d_in.data_ptr(), len(blob), ix, rs, d_out.data_ptr(), nbytes + 64)
        host = d_out[:got].cpu().numpy().tobytes()
        ok = got == total and all(zlib.crc32(host[o : o + e - b]) == zlib.crc32(data[b:e]) for (b, e), o in zip(rs, off))
        rmed, rlo, rhi = timed(lambda: codec.gzip_inflate_ranges_device(d_in.data_ptr(), len(blob), ix, rs, d_out.data_ptr(), nbytes + 64),
                               args.reps)
        _, touched = plan(x, rs)
        extra = ""
        if name.startswith("(c)"):
            extra = f"; {total / rmed / 1e9 / whole:.2f} x gzip_inflate_device's rate (target >= 0.9)"
        if name.startswith("(a)"):
            rate_a = len(rs) / rmed
        say(f"{name}: median {rmed * 1e3:.1f} ms, min {rlo * 1e3:.1f}, max {rhi * 1e3:.1f}; {len(rs) / rmed:.0f} ranges/s, "
            f"{total / rmed / 1e9:.2f} GB/s of output; {touched} touched chunks ({touched * 48 / 1024:.0f} MiB decoded){extra}; "
            f"output {'correct' if ok else 'WRONG'}")

    # single-core zlib from the same access points with the stored windows, on a sample of (a)
    sample = cases[0][1][: args.sample]
    by_pt = {c: w for c, w in x["points"]}
    ch = x["chunks"]
    ok = True
    where = [plan(x, [r])[0][0] for r in sample]     # (planned outside the timed loop)
    t0 = time.perf_counter()
    for (b, e), (p, last) in zip(sample, where):
        c, u, _ = ch[p]
        stop = ch[last + 1][0] if last + 1 < len(ch) else len(blob) - 8
        d = zlib.decompressobj(-15, zdict=by_pt[p]) if by_pt[p] else zlib.decompressobj(-15)
        out = d.decompress(blob[c:stop])
        ok = ok and out[b - u : e - u] == data[b:e]
    t = time.perf_counter() - t0
    cpu_rate = len(sample) / t
    say(f"zlib, one host core, from the same access points (sample of {len(sample)} ranges of (a)): {t / len(sample) * 1e3:.2f} ms per "
        f"range, {cpu_rate:.0f} ranges/s; output {'correct' if ok else 'WRONG'}")
    say(f"(a) against that baseline: {rate_a / cpu_rate:.1f} x (target >= 20)")
    codec.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
