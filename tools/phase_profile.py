"""Per-phase cycle counters of the compress kernel at a given level: python tools/phase_profile.py <level> [MiB] [fastq|sam]"""
import os, sys
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "7bgzf_b200"))
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "tests"))
import b200bgzf, helpers as H
level = int(sys.argv[1]); mib = int(sys.argv[2]) if len(sys.argv) > 2 else 64; kind = sys.argv[3] if len(sys.argv) > 3 else "fastq"
c = b200bgzf.Codec(0)
data = H.synth(kind, mib << 20)
c.compress(data[: 4 << 20], level)
c.profile(True, True)
out = c.compress(data, level)
prof = c.profile(False, True)
nblk = (mib << 20) / 0xff00
names = {0: "load", 1: "census", 2: "hash", 3: "peers", 10: "link", 21: "search: nearest", 4: "search: todo+deep", 15: "accept/dp", 5: "jump", 16: "walk clear+mark+list", 17: "walk a", 18: "walk b", 6: "walk c",
         7: "tally", 11: "sort (rank)", 12: "trees (+crc)", 13: "header", 8: "codes+tabs", 19: "sizes", 20: "scans", 14: "zero", 9: "emit"}
tot = sum(prof[k] for k in names)                 # (slots 22-27 hold the chain build / pass 1 details of tools/link_split.py, 28 the CRC tail)
print(f"level {level} {kind} {mib} MiB: ratio {len(out)/len(data):.4f}, {tot/nblk:.0f} cycles/block")
for k, v in sorted(names.items(), key=lambda kv: -prof[kv[0]]):
    print(f"  {v:24s} {prof[k]/nblk:10.0f}  {100*prof[k]/tot:5.1f}%")
# the CRC slices run beside the trees: cycles the CRC warps went on after the tree warps were done (0 = fully hidden)
print(f"  {'crc past trees':24s} {prof[28]/nblk:10.0f}")
