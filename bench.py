#!/usr/bin/env python
"""bench.py — BGZF compress & inflate GB/s (uncompressed) on B200, next to the reference's CPU path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--mib M] [--level L] [--kind fastq|sam] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...     (N > 1)
  python bench.py --impl reference ...      the reference's own CPU implementation (oracle/_ref), all host threads
  python bench.py --workload config3 [--gib 64] ...   BASELINE config 3: ONE 64 GiB SAM-like input, block ranges sharded over
                                            the ranks (strong scaling), shards joined at host-known offsets, whole-stream SHA-256

One "step" = one pass of the hot path over one batch: the whole workload (default 1 GiB of synthetic
FASTQ-like text cut into 0xff00-byte BGZF blocks, BGZF_METHOD=libdeflate6 class) compressed into one BGZF
stream; the inflate leg inflates that stream.  Every rank works on its own full-size batch (weak scaling);
blocks are independent, so there is no data-path collective — only the barrier and the max-over-ranks
reduction of the timing.
  value      device-resident compress throughput: input and output stay in HBM, CUDA events on the launch stream
  e2e        the same through the host-buffer C-ABI call (pinned host memory; H2D and D2H inside the timed region)
  inflate    the same two numbers for BGZF inflate of the stream just produced
  roofline   algorithmic bytes (payload read + stream written, SURVEY 8d) / device time, against the measured HBM peak
  cpu_baseline  the reference (oracle/_ref: the unmodified 7bgzf hook + libdeflate) on this box's host cores

--dump-outputs DIR writes, after the timed steps, what the last step of each timed leg handed its caller (see
dump_outputs).  The input is generated from a fixed seed, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "7bgzf_b200"))
BLOCK = 0xFF00


def load_gen():
    p = os.path.join(ROOT, "build", "libdatagen.so")
    if not os.path.exists(p):
        subprocess.run(["make", "-s", "testlibs"], cwd=ROOT, check=True)
    lib = ctypes.CDLL(p)
    lib.b200gen_fill.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_size_t]
    lib.b200gen_fill.restype = ctypes.c_size_t
    return lib


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region"""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.stop, self.index = [], threading.Event(), index
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.15)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(self.rows)}


def cpu_reference(args, data_addr, nbytes, kind_name, steps=1, warmup=0):
    """the reference's CPU path (unmodified hook + libdeflate, oracle/_ref) on a bounded sample, all host threads"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers as H
    if not H.have_ref():
        return None
    cores = os.cpu_count() or 1
    # levels 1-7 run the whole workload (about a second per GiB at level 6 on 16 cores); the slow levels are bounded to
    # roughly 10-20 s of CPU work per step (the reference's level 12 does ~1.2 MB/s per core)
    per_core = {8: 20e6, 9: 9e6, 10: 4e6, 11: 2e6, 12: 1.2e6}.get(args.level)
    sample = nbytes if per_core is None else int(min(nbytes, max(8 * BLOCK * cores, per_core * cores * 10)))
    if sample < nbytes:
        sample -= sample % BLOCK
    ref = H.Ref(args.level)
    nb = (sample + BLOCK - 1) // BLOCK
    sizes = (ctypes.c_uint32 * nb)()
    rc = ctypes.c_int()
    times = []
    # untimed warm-up on a small slice: the reference mallocs/frees its ~0.7 MB compressor per block, and the first
    # multi-threaded pass pays for the allocator's arena set-up
    H.oracle().refh_compress(ref.h, data_addr, min(sample, 16 * BLOCK * cores), BLOCK, cores, None, ctypes.addressof(sizes), ctypes.byref(rc))
    for i in range(warmup + steps):
        t = H.oracle().refh_compress(ref.h, data_addr, sample, BLOCK, cores, None, ctypes.addressof(sizes), ctypes.byref(rc))
        if i >= warmup:
            times.append(t)
    t = statistics.mean(times)
    out_bytes = sum(sizes)
    res = {"value": sample / t / 1e9, "unit": "GB/s", "cores": cores, "kind": "reference",
           "sample": f"{'the whole workload' if sample == nbytes else 'first'} {sample >> 20} MiB, reference bgzf_compress (BGZF_METHOD=libdeflate{args.level}) from {cores} pthreads over contiguous block ranges, memory to memory",
           "ratio": out_bytes / sample, "seconds": t}
    # inflate leg of the baseline: the reference's libdeflate decoder over the members it just could have written
    stream, _, _ = ref.compress_stream(ctypes.string_at(data_addr, min(sample, 64 << 20)), threads=cores)
    src = ctypes.create_string_buffer(stream, len(stream))
    out = ctypes.create_string_buffer(min(sample, 64 << 20))
    n, rc2 = ctypes.c_size_t(), ctypes.c_int()
    ti = min(H.oracle().refh_inflate(ref.h, ctypes.addressof(src), len(stream), cores, ctypes.addressof(out), len(out), ctypes.byref(n), ctypes.byref(rc2))
             for _ in range(3))
    res["inflate_value"] = n.value / ti / 1e9
    res["inflate_sample"] = f"{n.value >> 20} MiB, reference libdeflate_deflate_decompress per member from {cores} pthreads"
    return res


def bind_to_gpu_numa_node(index):
    """Multi-GPU boxes have two sockets: run this rank (and first-touch its pinned buffers) on the cores next to its
    GPU, or every host<->device copy of the end-to-end legs crosses the socket interconnect.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1 and 64 * i + b < ncpu}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def newest_traffic_file():
    """profiles/rNN_traffic.json of the latest round (ncu dram bytes per algorithmic byte, written by tools/traffic_from_ncu.py)"""
    import glob
    import re
    best = None
    for f in glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")):
        m = re.match(r"r(\d+)", os.path.basename(f))
        if m and (best is None or int(m.group(1)) > best[0]):
            best = (int(m.group(1)), f)
    return best[1] if best else None


def container_lines(codec, h_in, n, h_out, h_back):
    """whole-stream gzip (primed pieces), MiGz (512 KiB members), GZinga, dictzip, RAZF through b200bgzf_container_*_host:
    GB/s end to end (pinned host buffers, H2D + kernels + D2H + host framing in the timed call) and compressed size"""
    import torch
    import b200bgzf
    kinds = (("gzip", b200bgzf.CONTAINER_GZIP), ("migz", b200bgzf.CONTAINER_MIGZ), ("gzinga", b200bgzf.CONTAINER_GZINGA),
             ("dictzip", b200bgzf.CONTAINER_DICTZIP), ("razf", b200bgzf.CONTAINER_RAZF))
    res = {"MiB": n >> 20, "level": 6, "unit": "GB/s"}
    got = ctypes.c_size_t()
    for name, kind in kinds:
        cap = codec.lib.b200bgzf_container_bound(kind, 0, n)
        if cap > h_out.numel():
            continue

        def comp():
            rc = codec.lib.b200bgzf_container_compress_host(codec.h, kind, 0, h_in.data_ptr(), n, 6, h_out.data_ptr(), h_out.numel(), ctypes.byref(got))
            assert rc == 0, rc

        comp()
        t0 = time.perf_counter(); comp(); tc = time.perf_counter() - t0
        clen = got.value
        entry = {"compress_e2e": round(n / tc / 1e9, 2), "ratio": round(clen / n, 4)}
        if kind != b200bgzf.CONTAINER_GZIP:          # (a gzip member has no index: one warp decodes it)
            def dec():
                rc = codec.lib.b200bgzf_container_inflate_host(codec.h, kind, h_out.data_ptr(), clen, h_back.data_ptr(), n, ctypes.byref(got), 0)
                assert rc == 0 and got.value == n, (rc, got.value)

            dec()
            t0 = time.perf_counter(); dec(); td = time.perf_counter() - t0
            entry["inflate_e2e"] = round(n / td / 1e9, 2)
            entry["roundtrip_ok"] = bool(torch.equal(h_back[:n], h_in[:n]))
        res[name] = entry
    return res


DUMP_SAMPLE = 2 << 20          # bytes kept of each byte output; 4 of them as float32 plus the member sizes stay under 64 MB
DUMP_WINDOW = 4096


def member_sizes(stream):
    """compressed size of every member of a BGZF stream, by walking BSIZE (the EOF block included)"""
    sizes, off = [], 0
    while off + 18 <= len(stream):
        size = int(stream[off + 16]) + (int(stream[off + 17]) << 8) + 1
        sizes.append(size)
        off += size
    assert off == len(stream), "the BSIZE chain does not end at the end of the stream"
    return sizes


def dump_outputs(path, outputs):
    """Writes every (name, numpy array) as <path>/<name>.npy: byte arrays in float32, integer lists in float64.  A byte
    array longer than DUMP_SAMPLE is reduced to DUMP_SAMPLE bytes: whole DUMP_WINDOW-byte windows at offsets drawn from a
    fixed seed, in order, so that equal outputs give equal samples.  The bytes after the last whole window are not in the
    sample; of the compressed stream, compress_member_bytes covers every member, the EOF block included."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in outputs:
        if a.dtype == np.uint8:
            if a.size > DUMP_SAMPLE:
                rng = np.random.default_rng(0)
                starts = np.sort(rng.choice(a.size // DUMP_WINDOW, DUMP_SAMPLE // DUMP_WINDOW, replace=False)) * DUMP_WINDOW
                a = a[(starts[:, None] + np.arange(DUMP_WINDOW)).ravel()]
            a = a.astype(np.float32)
        else:
            a = a.astype(np.float64)
        np.save(os.path.join(path, f"{name}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps of each leg (default: 5; config3: 1, each a pass over the whole input); "
                                                            "the pageable-host legs run min(2, K) and report their own count; not for config5")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config1", choices=["config1", "config3", "config5"])
    ap.add_argument("--mib", type=int, default=1024, help="payload MiB per rank (BASELINE: 1 GiB)")
    ap.add_argument("--gib", type=int, default=None, help="config3: total GiB of the one sharded input (default 64, as BASELINE); "
                                                           "config5: GiB streamed through the hook (default 16)")
    ap.add_argument("--level", type=int, default=6)
    ap.add_argument("--kind", default="fastq", choices=["fastq", "sam"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-containers", action="store_true", help="skip the extra lines for the other containers (SURVEY 8f)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the outputs of each timed leg's last step "
                                                          "as DIR/<name>.npy (config1, --impl b200)")
    args = ap.parse_args()
    if args.workload == "config5" and args.steps is not None:
        ap.error("--steps is not for config5: it times one pass per caller count (three at 32 and 64 callers)")
    if args.steps is None:
        args.steps = 1 if args.workload == "config3" else 5
    if args.gib is None:
        args.gib = 16 if args.workload == "config5" else 64
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "config1" or args.impl != "b200"):
        ap.error("--dump-outputs is for --workload config1 --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload == "config3":
        args.kind = "sam"
    nbytes = args.mib << 20
    config = {"workload": f"{args.mib} MiB synthetic {args.kind.upper()}-like text (SURVEY App. B, seed {1 if args.kind == 'fastq' else 2}) per GPU, "
                          f"BGZF_METHOD=libdeflate{args.level} class, 0xff00-byte blocks; compress is the headline value, inflate of the same stream reported beside it",
              "block_bytes": BLOCK, "level": args.level, "bytes_per_gpu": nbytes, "parallelism": f"block-range sharding x{world}, no collective",
              "l2": f"inputs ({args.mib} MiB) are larger than the 126 MB L2; no explicit flush"}

    gen = load_gen()
    if args.workload == "config5":
        if rank == 0:
            run_config5(args)
        return
    if args.impl == "reference":
        # the reference's own CPU implementation on the SAME workload and warm-up as the GPU arm; rank 0 only
        if rank != 0:
            return
        buf = ctypes.create_string_buffer(nbytes)
        gen.b200gen_fill(0 if args.kind == "fastq" else 1, 1 if args.kind == "fastq" else 2, buf, nbytes)
        steps, warm = max(1, args.steps), max(0, args.warmup)
        r = cpu_reference(args, ctypes.addressof(buf), nbytes, args.kind, steps=steps, warmup=warm)
        if r is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/7bgzf_ref.so missing (run: make -f oracle/Makefile.ref)"}))
            return
        line = {"metric": "BGZF compress GB/s (uncompressed)", "value": r["value"], "unit": "GB/s", "n_gpus": args.gpus, "steps": steps,
                "warmup": warm, "ms_per_step": r["seconds"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic", "config": config, "impl": "reference",
                "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": r["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "inflate": {"value": r["inflate_value"], "unit": "GB/s", "sample": r["inflate_sample"]}, "ratio": r["ratio"]}
        print(json.dumps(line))
        return

    import hashlib
    import numpy as np
    import torch
    import torch.distributed as dist
    import b200bgzf

    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if numa:
        config["host_binding"] = f"each rank pinned to the {numa} cores of its GPU's NUMA node"
    if world > 1:
        # no collective on the data path (blocks are independent): the only exchanges are the barrier, the max-over-ranks
        # of the timings and the shard sizes, a few bytes over gloo
        dist.init_process_group("gloo")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(x):
        return reduce(x, dist.ReduceOp.MAX) if world > 1 else x

    def sum_over_ranks(x):
        return reduce(x, dist.ReduceOp.SUM) if world > 1 else x

    def gather_strings(sv):
        if world == 1:
            return [sv]
        out = [None] * world
        dist.all_gather_object(out, sv)
        return out

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)"
    traffic, traffic_file = {}, newest_traffic_file()
    try:
        traffic = json.load(open(traffic_file))
    except Exception:
        pass
    traffic_src = (f"{os.path.relpath(traffic_file, ROOT)} (ncu dram__bytes_read+write per algorithmic byte of one --set full capture) x this launch's algorithmic bytes"
                   if traffic else None)

    codec = b200bgzf.Codec(local_rank)
    stream = torch.cuda.current_stream()
    if args.workload == "config3":
        run_config3(args, codec, gen, rank, local_rank, world, barrier, max_over_ranks, sum_over_ranks, gather_strings, config, peak, peak_src, stream)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        codec.close()
        return

    h_in = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    gen.b200gen_fill(0 if args.kind == "fastq" else 1, 1 if args.kind == "fastq" else 2, h_in.data_ptr(), nbytes)
    bound = codec.bound(nbytes)
    # (room for the containers' extra lines too: their pieces are smaller than BGZF blocks, so their worst case is a little larger)
    h_out = torch.empty(max(bound, max(codec.lib.b200bgzf_container_bound(k, 0, nbytes) for k in range(1, 6))), dtype=torch.uint8, pin_memory=True)
    h_back = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    d_in = h_in.cuda()
    d_out = torch.empty(bound, dtype=torch.uint8, device="cuda")
    d_back = torch.empty(nbytes, dtype=torch.uint8, device="cuda")

    def run_timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        l0 = codec.launches()
        t0 = time.perf_counter()
        for a, b in evs:
            a.record(stream)
            fn()
            b.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        launches = codec.launches() - l0
        barrier()
        dev_ms = sum(a.elapsed_time(b) for a, b in evs)
        return dev_ms / 1e3, wall, launches

    with ClockSampler(local_rank) as clk:
        # --- compress, device resident: input/output stay in HBM; events on the stream the kernels run on
        clen = [0]

        def comp_dev():
            clen[0] = codec.compress_device(d_in.data_ptr(), nbytes, d_out.data_ptr(), bound, args.level, stream=stream.cuda_stream)

        t_dev, _, launches_c = run_timed(comp_dev, args.steps, args.warmup)
        clen_dev = clen[0]
        # --- inflate, device resident (member index built on the device inside the timed call)
        def inf_dev():
            codec.inflate_device(d_out.data_ptr(), clen[0], d_back.data_ptr(), nbytes, stream=stream.cuda_stream)

        t_idev, _, launches_i = run_timed(inf_dev, args.steps, args.warmup)
        # --- end to end through the host-buffer C ABI (pinned host memory, copies inside the timed region)
        def comp_e2e():
            clen[0] = codec.compress_into(h_in.data_ptr(), nbytes, h_out.data_ptr(), bound, args.level)

        _, w_e2e, _ = run_timed(comp_e2e, args.steps, args.warmup)
        clen_e2e = clen[0]

        def inf_e2e():
            codec.inflate_into(h_out.data_ptr(), clen[0], h_back.data_ptr(), nbytes)

        _, w_ie2e, _ = run_timed(inf_e2e, args.steps, args.warmup)
        ok = bool(torch.equal(d_back, d_in)) and bool(torch.equal(h_back, h_in))
        # --- the same calls on PAGEABLE host memory (what a caller that knows nothing of CUDA hands over)
        p_in = np.empty(nbytes, dtype=np.uint8)
        p_in[:] = h_in.numpy()
        p_out = np.empty(bound, dtype=np.uint8)
        p_out[:] = 0                                             # (touch the pages: not part of the measurement)
        psteps = max(1, min(2, args.steps))

        def comp_pg():
            clen[0] = codec.compress_into(p_in.ctypes.data, nbytes, p_out.ctypes.data, bound, args.level)

        _, w_pg, _ = run_timed(comp_pg, psteps, 1)
        ok = ok and bool(np.array_equal(p_out[: clen[0]], h_out.numpy()[: clen[0]]))
        p_back = np.empty(nbytes, dtype=np.uint8)
        p_back[:] = 0

        def inf_pg():
            codec.inflate_into(p_out.ctypes.data, clen[0], p_back.ctypes.data, nbytes)

        _, w_ipg, _ = run_timed(inf_pg, psteps, 1)
        ok = ok and bool(np.array_equal(p_back, p_in))
        del p_in, p_out, p_back

    if args.dump_outputs and rank == 0:
        stream_dev = d_out[:clen_dev].cpu().numpy()
        dump_outputs(args.dump_outputs, [("compress_stream", stream_dev),
                                         ("compress_member_bytes", np.array(member_sizes(stream_dev))),
                                         ("inflate_output", d_back.cpu().numpy()),
                                         ("compress_e2e_stream", h_out.numpy()[:clen_e2e]),
                                         ("inflate_e2e_output", h_back.numpy())])
    sha = hashlib.sha256(h_out.numpy()[: clen[0]]).hexdigest()          # the whole BGZF stream this rank produced (EOF included)
    shas = gather_strings(sha)
    steps = args.steps
    t_dev_m, t_idev_m = max_over_ranks(t_dev), max_over_ranks(t_idev)
    w_e2e_m, w_ie2e_m = max_over_ranks(w_e2e), max_over_ranks(w_ie2e)
    w_pg_m, w_ipg_m = max_over_ranks(w_pg), max_over_ranks(w_ipg)
    total_in = sum_over_ranks(float(nbytes))
    total_out = sum_over_ranks(float(clen[0]))
    tr_c = traffic.get("compress", {}).get("dram_per_algorithmic_byte")
    tr_i = traffic.get("inflate", {}).get("dram_per_algorithmic_byte")
    if rank == 0:
        value = total_in * steps / t_dev_m / 1e9
        alg_bytes = (nbytes + clen[0]) * steps         # per rank: payload read + stream written (SURVEY 8d)
        ach = alg_bytes / t_dev / 1e9
        ach_i = alg_bytes / t_idev / 1e9
        line = {
            "metric": "BGZF compress GB/s (uncompressed)", "value": value, "unit": "GB/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
            "ms_per_step": t_dev_m / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": config, "impl": "b200", "roundtrip_ok": ok,
            "ratio": total_out / total_in,
            "stream_sha256": sha, "stream_sha256_same_on_all_ranks": all(x == sha for x in shas),
            "e2e": {"value": total_in * steps / w_e2e_m / 1e9, "unit": "GB/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": clen[0],
                    "api": "b200bgzf_compress_host (pinned host buffers)"},
            "e2e_pageable": {"value": total_in * psteps / w_pg_m / 1e9, "unit": "GB/s", "steps": psteps,
                             "api": "b200bgzf_compress_host (pageable host buffers: malloc'ed numpy arrays)",
                             "inflate_value": total_in * psteps / w_ipg_m / 1e9},
            "inflate": {"value": total_in * steps / t_idev_m / 1e9, "unit": "GB/s", "ms_per_step": t_idev_m / steps * 1e3,
                        "e2e": {"value": total_in * steps / w_ie2e_m / 1e9, "unit": "GB/s", "h2d_bytes_per_step": clen[0], "d2h_bytes_per_step": nbytes,
                                "api": "b200bgzf_inflate_host (pinned host buffers)"},
                        "roofline": {"bound": "hbm", "achieved": ach_i, "peak": peak, "unit": "GB/s", "frac": ach_i / peak,
                                     "traffic": int(tr_i * (nbytes + clen[0])) if tr_i else None, "traffic_source": traffic_src,
                                     "kernel": "bgzf_inflate_kernel (+ member index kernels, <1% of the step)"}},
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": int(tr_c * (nbytes + clen[0])) if tr_c else None, "traffic_source": traffic_src,
                         "kernel": "bgzf_compress_kernel (+ scan/gather compaction, <1% of the step)", "peak_source": peak_src,
                         "algorithmic_bytes_per_step": nbytes + clen[0]},
            "gpu_launches": launches_c + launches_i,
            "clocks": clk.summary(),
        }
        if world == 1 and args.level == 6 and not args.no_containers:
            # SURVEY 8f ranks 3 / 4 on the same kernels (piece mode): the other containers end to end from the same pinned input
            # one timed call each after a warm-up; tools/container_bench.py has the reference's applets beside them
            try:
                line["containers"] = container_lines(codec, h_in, nbytes, h_out, h_back)
            except Exception as e:  # an extra: it must never sink the measurement
                line["containers"] = {"error": repr(e)}
        if not args.no_cpu_baseline:
            try:
                cb = cpu_reference(args, h_in.data_ptr(), nbytes, args.kind)
                if cb:
                    line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
                    line["cpu_baseline"]["inflate_value"] = cb["inflate_value"]
                    line["cpu_baseline"]["ratio"] = cb["ratio"]
            except Exception as e:  # the baseline must never sink the measurement
                line["cpu_baseline"] = {"error": repr(e)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    codec.close()


def run_config5(args):
    """BASELINE config 5: the LD_PRELOAD drop-in.  samtools/htslib are not on this image, so htslib's thread pool is played
    by build/hook_mt (tools/hook_mt.c): N pthreads, each a synchronous bgzf_compress(dst, &dlen, src, <= 0xff00, level) call
    at a time over BAM-encoded records (tools/datagen.c kind 2: what htslib hands the hook when samtools writes BAM) —
    --gib GiB streamed as repeats of a 1 GiB buffer.  The same harness drives the reference's 7bgzf.so on the host cores."""
    gib = args.gib
    path = "/dev/shm/b200bgzf_bam1g.bin"
    subprocess.run(f"{os.path.join(ROOT, 'build', 'datagen')} bam {1 << 30} 2 > {path}", shell=True, check=True)
    env = dict(os.environ, BGZF_METHOD=f"libdeflate{args.level}")
    ours, ref = os.path.join(ROOT, "7bgzf_b200", "7bgzf.so"), os.path.join(ROOT, "oracle", "_ref", "7bgzf_ref.so")

    def run(so, threads, repeat):
        out = subprocess.run([os.path.join(ROOT, "build", "hook_mt"), so, str(threads), path, str(repeat)], capture_output=True, text=True, env=env)
        return json.loads(out.stdout.strip().splitlines()[-1]) if out.returncode == 0 and out.stdout.strip() else {"error": out.stderr[-300:]}

    rows, cores = {}, os.cpu_count() or 1
    for th in (8, 16, 32, 64):
        runs = [run(ours, th, gib) for _ in range(3 if th >= 32 else 1)]
        vals = sorted(r["MB_per_s"] / 1e3 for r in runs if "MB_per_s" in r)
        if vals:
            rows[str(th)] = {"GBps": vals[len(vals) // 2], "runs": vals, "spread": (vals[-1] - vals[0]) / vals[len(vals) // 2], "ratio": runs[0].get("ratio")}
        else:
            rows[str(th)] = runs[0]
    refrows = {}
    if os.path.exists(ref):
        for th in (16, 64):
            r = run(ref, th, 1)
            refrows[str(th)] = {"GBps": r.get("MB_per_s", 0) / 1e3, "ratio": r.get("ratio")}
    os.unlink(path)
    best = max((v["GBps"], k) for k, v in rows.items() if "GBps" in v)
    line = {"metric": "BGZF compress GB/s (uncompressed) through the bgzf_compress() hook", "value": best[0], "unit": "GB/s", "n_gpus": 1, "steps": 1, "warmup": 1,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "impl": "b200",
            "config": {"workload": f"BASELINE config 5: {gib} GiB of BAM-encoded records (1 GiB synthetic buffer x {gib}) through LD_PRELOAD-style bgzf_compress calls, "
                                   f"one <= 0xff00-byte block per call, BGZF_METHOD=libdeflate{args.level}; htslib's pool emulated by build/hook_mt (samtools is not on the image)",
                       "callers_at_value": int(best[1]), "host_cores": cores},
            "callers": rows, "e2e": {"value": best[0], "unit": "GB/s", "h2d_bytes_per_step": gib << 30, "d2h_bytes_per_step": None,
                                     "api": "bgzf_compress (7bgzf.so), host buffers, synchronous per block"},
            "cpu_baseline": {"kind": "reference", "cores": cores, "unit": "GB/s", "value": max([v["GBps"] for v in refrows.values()] or [0]),
                             "callers": refrows, "sample": "1 GiB of the same records through the reference's 7bgzf.so from the same harness"}}
    print(json.dumps(line))


def run_config3(args, codec, gen, rank, local_rank, world, barrier, max_over_ranks, sum_over_ranks, gather_strings, config, peak, peak_src, stream):
    """BASELINE config 3: ONE input of --gib GiB SAM-like text (the concatenation of 1 GiB pieces, seeds 2, 3, ...), cut into
    0xff00-byte blocks; rank g of G takes blocks [B*g/G, B*(g+1)/G) (b200bgzf_shard_blocks), compresses them in 1 GiB
    chunks, and the shards are written at host-known offsets into one stream whose SHA-256 rank 0 reports: strong scaling,
    no collective on the data path.  A step is one pass over the whole input; the timed region of a chunk holds only the
    codec call (device-resident: kernels; end to end: H2D + kernels + D2H), never the generation of the input."""
    import hashlib
    import numpy as np
    import torch
    import b200bgzf
    from concurrent.futures import ThreadPoolExecutor

    PIECE = 1 << 30
    total = args.gib << 30
    nb = (total + BLOCK - 1) // BLOCK
    b0, b1 = b200bgzf.shard_blocks(nb, rank, world)
    lo, hi = b0 * BLOCK, min(b1 * BLOCK, total)
    mine = hi - lo
    # this rank's share of the input, generated piece by piece on the host cores (untimed)
    host = np.empty(max(mine, 1), dtype=np.uint8)
    pieces = range(lo // PIECE, (max(hi, lo + 1) - 1) // PIECE + 1) if mine else []

    def fill(i):
        buf = np.empty(PIECE, dtype=np.uint8)
        gen.b200gen_fill(1, 2 + i, buf.ctypes.data, PIECE)
        s, e = max(lo, i * PIECE), min(hi, (i + 1) * PIECE)
        host[s - lo : e - lo] = buf[s - i * PIECE : e - i * PIECE]

    with ThreadPoolExecutor(max(1, min(len(os.sched_getaffinity(0)), 16))) as ex:
        list(ex.map(fill, pieces))
    CH = 16384 * BLOCK                                            # chunk: 16384 blocks, just under 1 GiB
    bound = codec.bound(CH)
    h_in = torch.empty(CH, dtype=torch.uint8, pin_memory=True)
    h_out = torch.empty(bound, dtype=torch.uint8, pin_memory=True)
    d_in = torch.empty(CH, dtype=torch.uint8, device="cuda")
    d_out = torch.empty(bound, dtype=torch.uint8, device="cuda")
    shard = np.empty(int(mine * 0.30) + (1 << 20), dtype=np.uint8)   # this rank's part of the stream (SAM-like text: ratio ~0.13)
    steps = args.steps
    t_dev = t_e2e = 0.0
    launches = 0
    with ClockSampler(local_rank) as clk:
        # warm-up: the first chunk, args.warmup times through both paths
        n0 = min(CH, mine)
        if n0:
            h_in[:n0] = torch.from_numpy(host[:n0])
            d_in[:n0].copy_(h_in[:n0])
            for _ in range(args.warmup):
                codec.compress_device(d_in.data_ptr(), n0, d_out.data_ptr(), bound, args.level, eof=False, stream=stream.cuda_stream)
                codec.compress_into(h_in.data_ptr(), n0, h_out.data_ptr(), bound, args.level, eof=False)
        barrier()
        # every rank runs the same number of chunk turns and the ranks enter each timed call together (barrier), so that the
        # end-to-end leg sees the host side as it is when all GPUs copy at once
        nturns = int(max_over_ranks(float((mine + CH - 1) // CH)))
        for step in range(steps):
            pos = 0
            for turn in range(nturns):
                off = turn * CH
                n = min(CH, mine - off) if off < mine else 0
                if n:
                    h_in[:n] = torch.from_numpy(host[off : off + n])     # staging into pinned memory: untimed
                    d_in[:n].copy_(h_in[:n])
                barrier()
                if n:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    l0 = codec.launches()
                    e0.record(stream)
                    codec.compress_device(d_in.data_ptr(), n, d_out.data_ptr(), bound, args.level, eof=False, stream=stream.cuda_stream)
                    e1.record(stream)
                    torch.cuda.synchronize()
                    launches += codec.launches() - l0
                    t_dev += e0.elapsed_time(e1) / 1e3
                barrier()
                if n:
                    t0 = time.perf_counter()
                    clen = codec.compress_into(h_in.data_ptr(), n, h_out.data_ptr(), bound, args.level, eof=False)
                    t_e2e += time.perf_counter() - t0
                    if step == 0:
                        shard[pos : pos + clen] = h_out.numpy()[:clen]
                        pos += clen
            if step == 0:
                shard_len = pos if mine else 0
        barrier()
    # host-known offsets: every rank learns all shard sizes, writes its shard into ONE stream, rank 0 appends the EOF marker
    sizes = [int(x) for x in gather_strings(str(shard_len if mine else 0))]
    offs = [sum(sizes[:r]) for r in range(world)]
    path = f"/dev/shm/b200bgzf_config3_{os.environ.get('MASTER_PORT', '0')}.bgz"
    stream_len = sum(sizes) + 28
    if rank == 0:
        with open(path, "wb") as f:
            f.truncate(stream_len)
    barrier()
    mm = np.memmap(path, dtype=np.uint8, mode="r+")
    mm[offs[rank] : offs[rank] + sizes[rank]] = shard[: sizes[rank]]
    if rank == 0:
        mm[stream_len - 28 :] = np.frombuffer(b200bgzf.EOF_BLOCK, dtype=np.uint8)
    mm.flush()
    del mm
    barrier()
    t_dev_m, t_e2e_m = max_over_ranks(t_dev), max_over_ranks(t_e2e)
    if rank == 0:
        h = hashlib.sha256()
        check_ok, nm, usum = True, 0, 0
        with open(path, "rb") as f:
            while True:
                b = f.read(64 << 20)
                if not b:
                    break
                h.update(b)
        # spot check of the joined stream: the members around every shard boundary inflate to the input bytes they carry
        mm = np.memmap(path, dtype=np.uint8, mode="r")
        for r in range(world):
            if sizes[r] == 0:
                continue
            o = offs[r]
            msz = int(mm[o + 16]) + (int(mm[o + 17]) << 8) + 1
            first_block = b200bgzf.shard_blocks(nb, r, world)[0]
            member = bytes(mm[o : o + msz])
            want_lo = first_block * BLOCK
            piece = np.empty(PIECE, dtype=np.uint8)
            gen.b200gen_fill(1, 2 + want_lo // PIECE, piece.ctypes.data, PIECE)
            got = codec.inflate(member)
            exp = bytes(piece[want_lo % PIECE : want_lo % PIECE + len(got)])
            if len(exp) < len(got):                                  # the block straddles two pieces
                gen.b200gen_fill(1, 3 + want_lo // PIECE, piece.ctypes.data, PIECE)
                exp += bytes(piece[: len(got) - len(exp)])
            check_ok = check_ok and got == exp and len(got) == min(BLOCK, total - want_lo)
        del mm
        os.unlink(path)
        config = dict(config, workload=f"BASELINE config 3: ONE {args.gib} GiB synthetic SAM-like input (1 GiB pieces, seeds 2..{1 + args.gib}), libdeflate{args.level} class, "
                                       f"0xff00-byte blocks, block ranges [B*g/G, B*(g+1)/G) over {world} GPU(s), shards joined at host-known offsets",
                      bytes_total=total, bytes_per_gpu=None, chunk_bytes=CH,
                      step="one pass over the whole input in 1 GiB chunks; per chunk only the codec call is timed (CUDA events / wall clock), all ranks entering each timed call together (barrier); summed per rank, max over ranks")
        alg = (total + sum(sizes)) * steps
        line = {"metric": "BGZF compress GB/s (uncompressed)", "value": total * steps / t_dev_m / 1e9, "unit": "GB/s", "n_gpus": world, "steps": steps,
                "warmup": args.warmup, "ms_per_step": t_dev_m / steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
                "data": "synthetic", "config": config, "impl": "b200", "ratio": sum(sizes) / total,
                "stream_bytes": stream_len, "stream_sha256": h.hexdigest(), "shard_bytes": sizes, "boundary_members_ok": check_ok,
                "e2e": {"value": total * steps / t_e2e_m / 1e9, "unit": "GB/s", "h2d_bytes_per_step": total // world, "d2h_bytes_per_step": sum(sizes) // world,
                        "api": "b200bgzf_compress_host (pinned host buffers), one call per 1 GiB chunk"},
                "roofline": {"bound": "hbm", "achieved": alg / world / t_dev_m / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / world / t_dev_m / 1e9 / peak,
                             "traffic": None, "kernel": "bgzf_compress_kernel", "peak_source": peak_src},
                "gpu_launches": launches, "clocks": clk.summary()}
        print(json.dumps(line))


if __name__ == "__main__":
    main()
