"""Where the chain build and pass 1 spend their cycles: python tools/link_split.py [level ...] [--mib N] [--kind fastq|sam]

Per block (averaged over the blocks of one call), in cycles since the phase began:
  link            the whole chain build (producers + relay, to the barrier after it)
  last producer   the last producer warp has found the peers of its last tile
  last turn       the relay hands on the turn of the last tile (the ordered part is over)
  relay waits     per relay warp: spinning on ready[] (no tile from the producers yet) and on `turn` (waiting for the
                  relay warp before it)
  pass 1          the phase, and when its slowest and its fastest warp finish
and, for every 8th tile, when its ready flag went up and when the relay took its turn.
If the last producer finishes close to the end of the link phase, the producers bound it; if the turns trail the ready
flags by a growing margin, the relay's ordering does."""
import argparse, os, subprocess, sys
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "7bgzf_b200"))
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "tests"))
import b200bgzf, helpers as H

SLOTS, TURN, READY, LINKERS = 288, 32, 160, 4

ap = argparse.ArgumentParser()
ap.add_argument("levels", nargs="*", type=int, default=[1, 6])
ap.add_argument("--mib", type=int, default=64)
ap.add_argument("--kind", default="fastq")
args = ap.parse_args()

try:
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
except (OSError, subprocess.CalledProcessError):
    gpu = "unknown (nvidia-smi query failed)"
print(f"GPU 0: {gpu}")

c = b200bgzf.Codec(0)
data = H.synth(args.kind, args.mib << 20)
nblk = (args.mib << 20) / 0xff00
for level in args.levels:
    c.compress(data[: 4 << 20], level)
    c.profile(True, True, SLOTS)
    c.compress(data, level)
    p = [v / nblk for v in c.profile(False, True, SLOTS)]
    print(f"level {level} {args.kind} {args.mib} MiB: {sum(p[:22]):.0f} cycles/block")
    print(f"  link                  {p[10]:9.0f}")
    print(f"    last producer done  {p[22]:9.0f}  ({100 * p[22] / p[10]:.0f} % of link)")
    print(f"    last turn handed on {p[25]:9.0f}  ({100 * p[25] / p[10]:.0f} % of link)")
    print(f"    relay wait ready[]  {p[23] / LINKERS:9.0f}  per relay warp")
    print(f"    relay wait turn     {p[24] / LINKERS:9.0f}  per relay warp")
    print(f"  pass 1 (nearest)      {p[21]:9.0f}")
    print(f"    slowest warp done   {p[26]:9.0f}")
    print(f"    fastest warp done   {p[27]:9.0f}")
    print("  tile   ready    turn  turn-ready")
    for k in list(range(0, 128, 8)) + [111, 112, 127]:
        print(f"  {k:4d} {p[READY + k]:7.0f} {p[TURN + k]:7.0f} {p[TURN + k] - p[READY + k]:7.0f}")
c.close()
