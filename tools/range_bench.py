"""Random access on one GPU: b200bgzf_inflate_ranges_device over a 1 GiB FASTQ-like level-6 stream resident on the device
(larger than L2), against b200bgzf_inflate_device of the whole stream and single-core zlib on the same touched members.

  python tools/range_bench.py [--gib 1] [--reps 10] [--out FILE]

Workloads: (a) 1000 random 4 KiB ranges, (b) 1000 random 1 MiB ranges, (c) one 512 MiB range, each also as BGZF virtual
offsets.  Per workload: call time (host clock around the call, which synchronises; it includes the device index of the
stream, the planning and the copies of the range list), ranges/s, output GB/s and decoded-member GB/s = distinct touched
members x ISIZE / time (computed here from the member index).  The card's name and power limit are read in the same run.
"""
import argparse
import bisect
import ctypes
import os
import random
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "7bgzf_b200"), os.path.join(ROOT, "tests")]
import b200bgzf  # noqa: E402
import helpers as H  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return f"nvidia-smi unavailable ({e})"


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
    codec = b200bgzf.Codec(0)
    h_in = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    H._gen().b200gen_fill(0, 1, h_in.data_ptr(), nbytes)
    d_raw = h_in.cuda()
    d_stream = torch.empty(codec.bound(nbytes), dtype=torch.uint8, device="cuda")
    clen = codec.compress_device(d_raw.data_ptr(), nbytes, d_stream.data_ptr(), d_stream.numel(), 6)
    stream = d_stream[:clen].cpu().numpy().tobytes()
    c, u = b200bgzf.index(stream)
    total = nbytes
    isz = [(u[m + 1] if m + 1 < len(u) else total) - u[m] for m in range(len(u))]
    say(f"input: {nbytes} bytes FASTQ-like, level 6 -> {clen} bytes, {len(c)} members (device-resident, larger than the 126 MB L2)")
    d_out = torch.empty(nbytes + (64 << 20), dtype=torch.uint8, device="cuda")

    def timed(fn, reps):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        ts.sort()
        return ts[len(ts) // 2], ts[0], ts[-1]

    med, lo, hi = timed(lambda: codec.inflate_device(d_stream.data_ptr(), clen, d_out.data_ptr(), d_out.numel()), args.reps)
    whole_rate = total / med / 1e9
    say(f"inflate_device whole stream: {med * 1e3:.2f} ms median ({lo * 1e3:.2f}-{hi * 1e3:.2f}), {whole_rate:.2f} GB/s decoded")

    def voff(pos, at_end):
        """virtual offset of decoded position pos (at_end: an end position, so a member boundary names the member before)"""
        if pos == total:
            return len(stream) << 16
        m = bisect.bisect_right(u, pos) - 1
        while isz[m] == 0:
            m -= 1
        return (c[m] << 16) | (pos - u[m])

    rnd = random.Random(5)
    work = {
        "a: 1000 x 4 KiB": [(b, b + 4096) for b in (rnd.randrange(total - 4096) for _ in range(1000))],
        "b: 1000 x 1 MiB": [(b, b + (1 << 20)) for b in (rnd.randrange(total - (1 << 20)) for _ in range(1000))],
        "c: 1 x 512 MiB": [(total // 4, total // 4 + (512 << 20))] if total >= (768 << 20) else [(0, total // 2)],
    }
    say(f"{'workload':28s} {'call ms':>9s} {'ranges/s':>10s} {'out GB/s':>9s} {'decoded GB/s':>13s} {'members':>8s} {'zlib 1 core GB/s':>17s}")
    for name, ranges in work.items():
        touched = set()
        for b, e in ranges:
            touched.update(range(bisect.bisect_right(u, b) - 1, bisect.bisect_left(u, e)))
        dec = sum(isz[m] for m in touched)
        out = sum(e - b for b, e in ranges)
        # single-core zlib over the same members (once)
        t0 = time.perf_counter()
        for m in sorted(touched):
            end = c[m + 1] if m + 1 < len(c) else len(stream)
            zlib.decompressobj(-15).decompress(stream[c[m] + 18 : end - 8])
        tz = time.perf_counter() - t0
        for vo in (False, True):
            rr = [(voff(b, False), voff(e, True)) for b, e in ranges] if vo else ranges
            med, lo, hi = timed(lambda: codec.inflate_ranges_device(d_stream.data_ptr(), clen, rr, d_out.data_ptr(), d_out.numel(), voffsets=vo), args.reps)
            n, _ = codec.inflate_ranges_device(d_stream.data_ptr(), clen, rr, d_out.data_ptr(), d_out.numel(), voffsets=vo)
            assert n == out
            label = name + (" (voffsets)" if vo else "")
            say(f"{label:28s} {med * 1e3:9.2f} {len(ranges) / med:10.0f} {out / med / 1e9:9.2f} {dec / med / 1e9:13.2f} {len(touched):8d} {dec / tz / 1e9:17.3f}")
        say(f"{'':28s} (spread of the call time: {lo * 1e3:.2f}-{hi * 1e3:.2f} ms; decoded-member rate / whole-stream rate = {dec / med / 1e9 / whole_rate:.2f})")
    # correctness spot check of the last timed call against the host copy of the input
    got = d_out[:256].cpu().numpy().tobytes()
    b0 = work["c: 1 x 512 MiB"][0][0]
    assert got == h_in[b0 : b0 + 256].numpy().tobytes()
    codec.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
