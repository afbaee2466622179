"""Whole-stream gzip members without flush points on one GPU (DESIGN §6g): zlib -6, zlib -1 and GNU gzip -6 files of 1 GiB of
FASTQ-like data through b200bgzf_gzip_inflate_device (device-resident), b200bgzf_container_inflate_host (pinned buffers) and
`7gzip -d`, next to one warp on a 32 MiB slice and single-core zlib on the same file.

  python tools/gzip_search_bench.py [--gib 1] [--reps 10] [--out FILE] [--region-lib KIB=PATH ...]

Every GPU number is the median of `reps` calls after a warm-up, with min / max; every call synchronises and the host clock is
read around it; the files are larger than L2; every output's CRC-32 is checked.  Per-phase device times come from the kernel
records of torch.profiler (one profiled call per input, apart from the timed ones): the flush-point count and chain, the
search, the first boundary pass, the repair rounds, marker, anchor, resolve, narrow.  --region-lib times zlib -6 again with a
library built with another search region (make NVEXTRA=-DGZ_REGION=<bytes>), each in a process of its own.  The card's name
and power limit are read in the same run.
"""
import argparse
import ctypes
import os
import statistics
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "7bgzf_b200"), os.path.join(ROOT, "tests")]
import b200bgzf as B  # noqa: E402
import helpers as H  # noqa: E402

PHASES = [("count", ("gz_cand_scan_kernel", "bgzf_scan")), ("search", ("gz_search_kernel",)), ("bound", ("gz_bit_bound_kernel",)),
          ("marker", ("gz_bit_marker_kernel",)), ("prefix", ("gz_prefix_kernel",)), ("anchor", ("gz_anchor_kernel",)),
          ("resolve", ("gz_resolve_kernel",)), ("narrow", ("gz_narrow_kernel",))]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return f"nvidia-smi unavailable ({e})"


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), min(ts), max(ts)


def zlib_member(data, level):
    z = zlib.compressobj(level, zlib.DEFLATED, 31)
    return z.compress(data) + z.flush()


def gnu_gzip(data, level):
    return subprocess.run(["gzip", "-c", "-n", "-%d" % level], input=data, capture_output=True, check=True).stdout


def phases(codec, call):
    """device time per phase (ms) of one call, from the profiler's kernel records; the boundary pass split into its first
    launch and the repair rounds"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    ks = sorted((e.time_range.start, e.time_range.elapsed_us(), e.name) for e in prof.events()
                if e.device_type == torch.autograd.DeviceType.CUDA)
    out, rounds = {}, 0
    for _, us, name in ks:
        for ph, keys in PHASES:
            if any(k in name for k in keys):
                if ph == "bound":
                    rounds += 1
                    ph = "bound" if rounds == 1 else "repair"
                out[ph] = out.get(ph, 0.0) + us / 1e3
                break
        else:
            out["other (copies, memsets, verify)"] = out.get("other (copies, memsets, verify)", 0.0) + us / 1e3
    return out, max(rounds - 1, 0)


def device_rate(codec, blob, n, want_crc, d_out, reps, say, label):
    import torch
    d_in = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
    t0 = time.perf_counter()
    got = codec.gzip_inflate_device(d_in.data_ptr(), len(blob), d_out.data_ptr(), n + 64)
    first = time.perf_counter() - t0
    ok = got == n and zlib.crc32(d_out[:n].cpu().numpy().tobytes()) == want_crc
    if first > 5:
        say(f"  {label}gzip_inflate_device: {first:.1f} s for the first call (one warp); not repeated; "
            f"output {'correct' if ok else 'WRONG'}")
        return None
    before = codec.launches()
    call = lambda: codec.gzip_inflate_device(d_in.data_ptr(), len(blob), d_out.data_ptr(), n + 64)  # noqa: E731
    med, lo, hi = timed(call, reps)
    nl = (codec.launches() - before) // (reps + 1)
    say(f"  {label}gzip_inflate_device: median {med * 1e3:.1f} ms ({n / med / 1e9:.2f} GB/s, {n / med / 1e9 / 0.46:.1f} x 0.46 GB/s), "
        f"min {lo * 1e3:.1f}, max {hi * 1e3:.1f}; {nl} launches per call; output {'correct' if ok else 'WRONG'}")
    ph, rounds = phases(codec, call)
    say("  " + label + "phases (ms): " + ", ".join(f"{k} {v:.2f}" for k, v in ph.items()) + f"; repair rounds {rounds}")
    return med


def variant(args):
    """--blob: one file through a library of another region size (a process of its own)"""
    import torch
    blob = open(args.blob, "rb").read()
    n = int(args.gib * (1 << 30))
    codec = B.Codec(0, path=args.lib)
    d_out = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
    device_rate(codec, blob, n, args.crc, d_out, args.reps, lambda s: print(s, flush=True), f"[S = {args.kib} KiB] ")
    codec.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--region-lib", action="append", default=[], help="KIB=PATH: a library built with GZ_REGION = KIB KiB")
    ap.add_argument("--blob", help=argparse.SUPPRESS)
    ap.add_argument("--lib", help=argparse.SUPPRESS)
    ap.add_argument("--kib", help=argparse.SUPPRESS)
    ap.add_argument("--crc", type=int, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.blob:
        return variant(args)
    import torch

    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say(f"card: {card()}")
    nbytes = int(args.gib * (1 << 30))
    data = H.synth("fastq", nbytes)
    crc = zlib.crc32(data)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(3) as ex:
        jobs = [("zlib -6", ex.submit(zlib_member, data, 6)), ("zlib -1", ex.submit(zlib_member, data, 1)),
                ("GNU gzip -6", ex.submit(gnu_gzip, data, 6))]
        inputs = [(name, j.result()) for name, j in jobs]
    say(f"input: FASTQ-like {nbytes} B (generator seed 1); files built on the host in {time.perf_counter() - t0:.0f} s")
    codec = B.Codec(0)
    lib, h = codec.lib, codec.h
    lib.b200bgzf_host_alloc.restype = ctypes.c_void_p
    d_out = torch.empty(nbytes + 64, dtype=torch.uint8, device="cuda")
    for name, blob in inputs:
        say(f"--- {name}: {len(blob)} B -> {nbytes} B; flush patterns in it: {blob.count(bytes([0, 0, 255, 255]))}")
        if device_rate(codec, blob, nbytes, crc, d_out, args.reps, say, "") is None:
            continue
        p_in = lib.b200bgzf_host_alloc(len(blob))
        p_out = lib.b200bgzf_host_alloc(nbytes + 64)
        ctypes.memmove(p_in, blob, len(blob))
        cnt = ctypes.c_size_t()

        def host():
            rc = lib.b200bgzf_container_inflate_host(h, B.CONTAINER_GZIP, p_in, len(blob), p_out, nbytes + 64, ctypes.byref(cnt), 0)
            assert rc == 0, rc

        med, lo, hi = timed(host, args.reps)
        ok = zlib.crc32(ctypes.string_at(p_out, nbytes)) == crc
        say(f"  container_inflate_host (pinned): median {med * 1e3:.1f} ms ({nbytes / med / 1e9:.2f} GB/s), min {lo * 1e3:.1f}, "
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
            say(f"  7gzip -d: {t:.2f} s wall ({nbytes / t / 1e9:.2f} GB/s; target < 2 s), exit {r.returncode}, "
                f"stderr {r.stderr.decode().strip()!r}")
        t0 = time.perf_counter()
        out = zlib.decompress(blob, 31)
        t = time.perf_counter() - t0
        say(f"  zlib, one host core: {t:.2f} s ({nbytes / t / 1e9:.2f} GB/s); output {'correct' if zlib.crc32(out) == crc else 'WRONG'}")
        del out
    # one warp on a 32 MiB slice (zlib -6)
    sl = zlib_member(data[: 32 << 20], 6)
    units, total = B.container_units(B.CONTAINER_GZIP, sl)
    t0 = time.perf_counter()
    out = codec.inflate_units(sl, units, total)
    t = time.perf_counter() - t0
    say(f"one warp (inflate_units, 32 MiB zlib -6 slice): {t:.2f} s ({(32 << 20) / t / 1e6:.1f} MB/s); "
        f"output {'correct' if out == data[: 32 << 20] else 'WRONG'}")
    codec.close()
    del d_out
    torch.cuda.empty_cache()
    if args.region_lib:
        with tempfile.NamedTemporaryFile(suffix=".gz") as f:
            f.write(inputs[0][1])
            f.flush()
            for spec in args.region_lib:
                kib, path = spec.split("=", 1)
                say(f"--- zlib -6 with the search region at {kib} KiB ({path})")
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--blob", f.name, "--lib", path, "--kib", kib,
                                    "--crc", str(crc), "--gib", str(args.gib), "--reps", str(args.reps)],
                                   capture_output=True, text=True)
                for s in r.stdout.splitlines():
                    say(s)
                if r.returncode:
                    say(f"  failed: {r.stderr.strip()[-500:]}")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
