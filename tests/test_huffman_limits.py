"""The code-length limits of the compressor's three Huffman codes, and its degenerate trees, against the emulator.

DEFLATE caps litlen and distance codes at 15 bits and the precode at 7.  A tree deeper than that is clamped, and the
per-length counts are repaired (bg_huff_lengths, bg_phase_huff_fix; on the GPU warp_huff_lengths for the distance code and
the precode).  A dynamic block with no distance code used, or exactly one, takes the m < 2 special cases.  FASTQ/SAM-like
data reaches these branches only by chance, so the inputs here are built to reach them: seeded byte streams in which no
3-byte string repeats unless a copy is planted on purpose, so that every level's parser sees the same symbols.

The CPU tests prove through the emulator's tree statistics (H.emul_trees) that every case still reaches its branch at
every level: a change to a generator or to the parser that stops reaching one fails here.  The GPU tests compare the
kernel's bytes with the emulator's for the same cases.  `pytest -s -k table` prints the statistics."""
import functools
import os
import random
import subprocess
import sys
import zlib

import pytest

import b200bgzf
import helpers as H

LEVELS = range(1, 13)
# first distance of each DEFLATE distance code (RFC 1951 3.2.5)
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577, 32769]


def fib(k):
    """1, 1, 2, 3, 5, ...: the leaf weights of the deepest Huffman tree for their total"""
    a, b, out = 1, 1, []
    for _ in range(k):
        out.append(a)
        a, b = b, a + b
    return out


class Stream:
    """Bytes in which no 3-byte string occurs twice, except inside copies planted with copy(): no match of 3 bytes or
    more can start anywhere else."""

    def __init__(self, seed, alphabet=range(256)):
        self.r = random.Random(seed)
        self.alpha = list(alphabet)
        self.out, self.seen, self.fresh = bytearray(), set(), []

    def push(self, b, fresh=True):
        self.out.append(b)
        self.fresh.append(fresh)
        if len(self.out) >= 3:
            self.seen.add(bytes(self.out[-3:]))

    def new(self, b):
        return len(self.out) < 2 or bytes(self.out[-2:]) + bytes([b]) not in self.seen

    def noise(self, n):
        for _ in range(n):
            b = self.r.choice(self.alpha)
            while not self.new(b):
                b = self.r.choice(self.alpha)
            self.push(b)

    def try_copy(self, d, n):
        """plant a copy of n bytes from distance d if its source is unused noise of distinct bytes and no match could
        start before it (the 3-byte strings that reach into it are new).  The noise after it ends any match with it."""
        p = len(self.out)
        src = range(p - d, p - d + min(d, n))
        if not all(self.fresh[i] for i in src) or len({self.out[i] for i in src}) < len(src):
            return False
        c = bytes(self.out[p - d + i % d] for i in range(n))
        if bytes(self.out[-2:]) + c[:1] in self.seen or bytes(self.out[-1:]) + c[:2] in self.seen:
            return False
        for i in src:
            self.fresh[i] = False
        for b in c:
            self.push(b, False)
        return True


def litlen_deep(k, seed=1):
    """Litlen over 15 bits: noise over 200 byte values with k further byte values planted 1, 2, 3, 5, 8, ... times
    (with the end-of-block symbol's 1, a Fibonacci-weighted tail: a chain of k levels below the noise symbols)."""
    r = random.Random(seed)
    rare = [200 + j for j, c in enumerate(fib(k + 1)[1:]) for _ in range(c)]
    r.shuffle(rare)
    slots = set(r.sample(range(2, H.BLOCK), len(rare)))
    s = Stream(seed, range(200))
    owed = 0
    for p in range(H.BLOCK):
        owed += p in slots
        j = next((j for j in range(len(rare)) if s.new(rare[j])), None) if owed else None
        if j is None:
            s.noise(1)
        else:
            s.push(rare.pop(j))
            owed -= 1
    assert not rare
    return bytes(s.out)


def dist_copies(counts, seed=1):
    """Noise with planted copies: counts[c] copies at distances of DEFLATE distance code c, in a seeded order; 4-byte
    copies for the codes up to 5, 6-byte ones beyond (so that every level's parser takes them)."""
    r = random.Random(seed)
    ev = [c for c, m in counts.items() for _ in range(m)]
    r.shuffle(ev)
    s = Stream(seed)
    s.noise(4)
    while ev:
        assert len(s.out) < H.BLOCK - 8, "the copies do not fit one block"
        e = ev[-1]
        n = 4 if e <= 5 else 6
        lo, hi = DIST_BASE[e], min(DIST_BASE[e + 1] - 1, len(s.out))
        placed = lo <= hi and any(s.try_copy(r.randint(lo, hi), n) for _ in range(12))
        if placed:
            ev.pop()
        s.noise(r.randint(1, 2) if placed else 1)
    s.noise(H.BLOCK - len(s.out))
    return bytes(s.out)


def literal_lengths(nlen, seed=1, n=8000):
    """A block of literals only whose litlen code has nlen[L] symbols of L bits (byte values drawn at random, each with
    weight 2^-L): the precode, which codes these lengths, sees skewed counts spread over many lengths."""
    r = random.Random(seed)
    lens = [L for L, k in sorted(nlen.items()) for _ in range(k)]
    tot = sum(2.0 ** -L for L in lens)
    pool = [s for s, L in zip(r.sample(range(256), len(lens)), lens) for _ in range(max(1, round(n * 2.0 ** -L / tot)))]
    r.shuffle(pool)
    s = Stream(seed)
    while pool:
        j = r.randrange(len(pool))
        for _ in range(400):
            if s.new(pool[j]):
                break
            j = r.randrange(len(pool))
        s.push(pool[j])
        pool[j] = pool[-1]
        pool.pop()
    return bytes(s.out)


def de_bruijn(k, n):
    """every string of n symbols over k letters exactly once (cyclically): no 3-byte match for n = 3"""
    a, seq = [0] * k * n, []

    def db(t, p):
        if t > n:
            if n % p == 0:
                seq.extend(a[1 : p + 1])
        else:
            a[t] = a[t - p]
            db(t + 1, p)
            for j in range(a[t - p] + 1, k):
                a[t] = j
                db(t + 1, t)

    db(1, 1)
    return bytes(48 + x for x in seq)


# case -> (generator, what it reaches at every level: {tree: overflow}, {"dist_m": used distance codes},
#          {"<tree>_ties": (leaves of the weight of the leaf before them, leaf / merged-node ties of the merge)})
BELL = {4: 1, 5: 2, 6: 5, 7: 13, 8: 34, 9: 89, 10: 55, 11: 21, 12: 8, 13: 3, 14: 1}
CASES = {
    "litlen_ovf2": (lambda: litlen_deep(8), {"litlen": 2}),
    "litlen_ovf_large": (lambda: litlen_deep(12), {"litlen": 6}),
    "dist_ovf2": (lambda: dist_copies({2 + i: c for i, c in enumerate(fib(17)[::-1])}), {"dist": 2, "dist_m": 17}),
    "dist_ovf4": (lambda: dist_copies({1 + i: c for i, c in enumerate(fib(18)[::-1])}), {"dist": 4, "dist_m": 18}),
    "precode_ovf2": (lambda: literal_lengths(BELL, seed=8), {"precode": 2, "dist_m": 0}),
    "precode_ovf4": (lambda: literal_lengths({6: 6, 7: 6, 8: 14, 9: 35, 10: 55, 11: 78, 12: 27, 13: 26}, seed=376),
                     {"precode": 4, "dist_m": 0}),
    "precode_ovf6": (lambda: literal_lengths({6: 1, 7: 32, 8: 42, 9: 65, 10: 8, 11: 5, 12: 39, 13: 2}, seed=625),
                     {"precode": 6, "dist_m": 0}),
    "no_match_de_bruijn": (lambda: de_bruijn(40, 3), {"dist_m": 0}),
    "one_distance": (lambda: dist_copies({10: 400}), {"dist_m": 1}),
    # equal weights among the leaves and between leaves and merged nodes (the merge takes the leaf first)
    "dist_ties": (lambda: dist_copies({4: 8, 5: 8, 6: 8, 7: 8, 8: 16, 9: 16, 10: 32, 11: 1, 12: 1, 13: 2, 14: 2, 15: 4}),
                  {"dist_m": 12, "dist_ties": (6, 6)}),
    "precode_ties": (lambda: literal_lengths({6: 4, 7: 8, 8: 16, 9: 32, 10: 64, 11: 16, 12: 16, 13: 8, 14: 8}, seed=3, n=12000),
                     {"dist_m": 0, "precode_ties": (2, 2)}),
}


@functools.lru_cache(None)
def case(name):
    return CASES[name][0]()


def trees(data, level):
    rc, member = H.emul_block(data, level)
    assert rc == 0, rc
    return H.emul_trees(), member


@pytest.mark.parametrize("name", sorted(CASES))
def test_case_reaches_its_branch_at_every_level(name):
    data = case(name)
    assert len(data) <= H.BLOCK
    want = CASES[name][1]
    for level in LEVELS:
        t, _ = trees(data, level)
        assert t["btype"] == 2, (level, t)
        for tree, ovf in want.items():
            if tree == "dist_m":
                assert t["dist"][0] == ovf, (level, t)
            elif tree.endswith("_ties"):
                assert H.emul_ties()[tree[:-5]] == ovf, (level, H.emul_ties())
            else:
                assert t[tree][1] == ovf, (level, t)


def test_distance_overflow_in_two_cases_and_the_table():
    """prints, per case, BTYPE and (used symbols, overflow) of each tree at levels 1, 6 and 12, and the ties of the
    distance and precode trees"""
    with_dist = set()
    for name in sorted(CASES):
        row = []
        for level in (1, 6, 12):
            t, _ = trees(case(name), level)
            row.append("L%-2d btype %d litlen %-10s dist %-8s precode %s" % (level, t["btype"], t["litlen"], t["dist"], t["precode"]))
            if t["dist"][1]:
                with_dist.add(name)
        print("%-20s %s | ties %s" % (name, " | ".join(row), H.emul_ties()))
    assert len(with_dist) >= 2, with_dist


@pytest.mark.parametrize("level", LEVELS)
def test_statistics_give_the_type_of_the_emitted_block(level):
    """BTYPE of the statistics is that of the DEFLATE block the call wrote (its first byte after the 18-byte BGZF
    header): stored for noise, static for a few words, dynamic for a case"""
    for data, btype in ((H.lcg_noise(5000), 0), (b"the quick brown fox jumps over the lazy dog. " * 3, 1), (case("dist_ovf2"), 2)):
        t, member = trees(data, level)
        assert t["btype"] == btype == (member[18] >> 1) & 3, (level, t)


# ---- the same cases on the GPU ----

@pytest.fixture(scope="module")
def codec():
    c = b200bgzf.Codec(0)
    yield c
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_gpu_bit_exact_vs_emulator(codec, name):
    data = case(name)
    for level in LEVELS:
        got = codec.compress(data, level)
        assert got == H.emul_stream(data, level), level
        assert H.gunzip(got) == data
        assert codec.inflate(got, flags=b200bgzf.VERIFY) == data


SPLIT_LEVELS = (1, 4, 6, 9, 10)
SPLIT_DRIVER = r"""
import sys
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2])
import b200bgzf, test_huffman_limits as T
c = b200bgzf.Codec(0)
for level in T.SPLIT_LEVELS:
    for name in sorted(T.CASES):
        got, st = c.compress_blocks([T.case(name)], level)
        assert st == [0], (level, name, st)
        sys.stdout.buffer.write(got[0])
"""


@pytest.mark.gpu
def test_gpu_one_member_calls_on_a_cluster():
    """the one-block path that splits the search over a cluster of CTAs (B200BGZF_SPLIT, read once per process)"""
    want = b"".join(trees(case(name), level)[1] for level in SPLIT_LEVELS for name in sorted(CASES))
    for split in ("1", "8"):
        env = dict(os.environ, B200BGZF_SPLIT=split)
        r = subprocess.run([sys.executable, "-c", SPLIT_DRIVER, os.path.join(H.ROOT, "tests"), os.path.join(H.ROOT, "7bgzf_b200")],
                           capture_output=True, env=env)
        assert r.returncode == 0, r.stderr.decode()
        assert r.stdout == want, split


@pytest.mark.gpu
@pytest.mark.parametrize("level", [1, 6, 12])
def test_gpu_pieces_with_and_without_history(codec, level):
    """piece mode on the distance-overflow input: one final piece without history (the tree of the whole input, over 15
    bits), and two pieces of 32640 bytes where the second's matches may reach into the first (history 32640; each half
    has half the copies, so its distance tree stays within 15 bits)"""
    data = case("dist_ovf4")
    for hist, bs in ((0, H.BLOCK), (32640, 32640)):
        stream, off, crc = codec.compress_pieces(data, b200bgzf.PieceSpec(0xFFFFFFFF, 0, 0, 0, 0, 0, hist, 0), level, bs)
        want = b""
        for o in range(0, len(data), bs):
            m, _ = H.emul_piece(data[o : o + bs], level, final=o + bs >= len(data), history=data[max(0, o - hist) : o])
            want += m
            if hist == 0:
                assert H.emul_trees()["dist"][1] == 4
        assert stream == want, hist
        d = zlib.decompressobj(-15)
        assert d.decompress(stream) == data and d.eof
