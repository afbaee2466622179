"""GPU (B200): the parity tests proper.  Everything goes through the C ABI (lib7bgzf_b200.so / 7bgzf.so / the
7bgzf applet); the oracle (emulator of the block algorithm, oracle/liboracle.so, oracle/_ref) is only the checker."""
import ctypes
import json
import os
import struct
import subprocess
import sys
import threading
import zlib

import pytest

import b200bgzf
import helpers as H

pytestmark = pytest.mark.gpu
KA = json.load(open(os.path.join(H.GOLDEN, "known_answers.json")))
MAL = json.load(open(os.path.join(H.GOLDEN, "malformed.json")))


@pytest.fixture(scope="module")
def codec():
    c = b200bgzf.Codec(0)       # raises if the CUDA library / device is missing: no fallback
    yield c
    c.close()


EDGE = {
    "empty": b"", "A": b"A", "AB": b"AB", "zeros65280": bytes(65280), "noise65280": H.lcg_noise(65280), "acgt": H.acgt(65280),
    "n31": H.lcg_noise(31), "n32": H.lcg_noise(32), "x700": b"x" * 700, "text": (b"the quick brown fox jumps over the lazy dog. " * 2000)[:65280],
    "ragged": H.synth("sam", 3 * H.BLOCK + 17), "short_tail": H.synth("fastq", H.BLOCK + 5),
}


@pytest.mark.parametrize("name", sorted(EDGE))
@pytest.mark.parametrize("level", [1, 6, 12])
def test_edge_inputs_bit_exact_vs_emulator_and_decode(codec, name, level):
    data = EDGE[name]
    got = codec.compress(data, level)
    assert got == H.emul_stream(data, level)                  # same bytes as the CPU run of the same algorithm
    assert H.gunzip(got) == data
    rc, out, _ = H.oracle_decompress(got)
    assert rc == 0 and out == data
    assert codec.inflate(got) == data


def test_known_answers_of_the_reference(codec):
    for name, payload in (("A", b"A"), ("zeros65280", bytes(65280)), ("noise65280", H.lcg_noise(65280))):
        members, st = codec.compress_blocks([payload], 6)
        assert st == [0] and len(members[0]) == KA[f"{name}_L6"]["size"]
        crc, isize = struct.unpack("<II", members[0][-8:])
        assert "%08x" % crc == KA[f"{name}_L6"]["crc"] and isize == len(payload)
    members, _ = codec.compress_blocks([b"A"], 6)
    assert members[0].hex().startswith(KA["A_L6"]["head"])
    # 65536 payload bytes: zeros fit, noise cannot (reference returns 1 and leaves *dlen alone)
    members, st = codec.compress_blocks([bytes(65536), H.lcg_noise(65536)], 6)
    assert st == [0, 1] and len(members[0]) == KA["zeros65536_L6"]["size"] and members[1] is None
    assert H.gunzip(members[0]) == bytes(65536)
    # capacity conventions
    members, st = codec.compress_blocks([H.lcg_noise(1000)], 6, caps=[30])
    assert st == [1]


@pytest.mark.parametrize("kind", ["fastq", "sam"])
@pytest.mark.parametrize("level", list(range(1, 13)))
def test_stream_parity_size_crc_and_reference_decoder(codec, kind, level):
    """every level class against the reference at the SAME level: decodes through the reference's libdeflate decoder,
    CRC32/ISIZE exact, size within 3 % of the reference's (BASELINE north_star tolerance)"""
    data = H.synth(kind, (8 << 20) if level < 10 else (2 << 20))     # the reference's level 12 runs at ~1 MB/s per core
    got = codec.compress(data, level)
    assert got[: 20 * 16384].startswith(H.emul_stream(data[: 4 * H.BLOCK], level, eof=False))
    mem = H.members(got)
    assert got.endswith(H.EOF_BLOCK) and len(mem) == (len(data) + H.BLOCK - 1) // H.BLOCK + 1
    for i, (off, size, isize, crc) in enumerate(mem[:-1]):
        blk = data[i * H.BLOCK : (i + 1) * H.BLOCK]
        assert isize == len(blk) and crc == zlib.crc32(blk) and size <= 65536
    assert H.gunzip(got) == data
    if H.have_ref():
        ref = H.Ref(level)
        rc, out, _ = ref.inflate_stream(got)                       # the reference's own libdeflate decoder
        assert rc == 0 and out == data
        _, ref_sizes, _ = ref.compress_stream(data, keep=False, threads=os.cpu_count() or 1)
        assert len(got) - 28 <= 1.03 * sum(ref_sizes), (len(got), sum(ref_sizes))
    elif level in (1, 6, 12):
        # without the compiled reference: its committed stream of the first two blocks of the same input
        ref_mem = H.members(open(os.path.join(H.GOLDEN, f"ref_{kind}_L{level}.bgz"), "rb").read())
        assert sum(m[1] for m in mem[:2]) <= 1.03 * sum(m[1] for m in ref_mem), (mem[:2], ref_mem)
        assert [m[2:] for m in mem[:2]] == [m[2:] for m in ref_mem]          # ISIZE and CRC32 as the reference writes them


@pytest.mark.parametrize("kind", ["fastq", "sam"])
def test_whole_stream_bit_exact_vs_emulator(codec, kind):
    """every member of a 3 MiB stream equals the CPU run of the same block algorithm (exercises the chain build's
    ordering assumptions on run-heavy quality strings and overlapping reads, not just the first blocks)"""
    data = H.synth(kind, 3 << 20)
    for level in (6, 9):
        assert codec.compress(data, level) == H.emul_stream(data, level)


@pytest.mark.parametrize("level", [1, 6])
def test_bam_like_binary_records_bit_exact_vs_emulator(codec, level):
    """binary-looking blocks take the deeper chains (bg_phase_settle): same bytes as the CPU run, decodes, inflates"""
    data = H.bamlike(6 * H.BLOCK + 1234)
    got = codec.compress(data, level)
    assert got == H.emul_stream(data, level)
    assert H.gunzip(got) == data and codec.inflate(got, flags=b200bgzf.VERIFY) == data


def test_odd_block_sizes_and_unaligned_sources(codec):
    """payload blocks that are not multiples of 16 bytes (no TMA alignment) and tiny blocks"""
    data = H.synth("sam", 300000) + H.lcg_noise(777)
    for bs in (1, 17, 1000, 4099, 65535, 65536):
        d = data[: min(len(data), bs * 40)]
        got = codec.compress(d, 6, block_size=bs)
        assert got == H.emul_stream(d, 6, block=bs), bs
        assert codec.inflate(got) == d
    import torch
    # device API with a source pointer that is only byte aligned
    buf = torch.frombuffer(bytearray(b"\0" * 3 + data), dtype=torch.uint8).cuda()
    out = torch.empty(codec.bound(len(data)), dtype=torch.uint8, device="cuda")
    n = codec.compress_device(buf.data_ptr() + 3, len(data), out.data_ptr(), out.numel(), 6)
    assert bytes(out[:n].cpu().numpy()) == H.emul_stream(data, 6)


def test_reference_applet_decodes_gpu_stream(codec):
    if not os.path.exists(H.REF_7BGZF):
        pytest.skip("oracle/_ref not built")
    data = H.synth("sam", 2 << 20)
    r = subprocess.run([H.REF_7BGZF, "-d"], input=codec.compress(data, 6), capture_output=True)
    assert r.returncode == 0 and r.stdout == data


def test_deterministic_across_runs_batches_and_paths(codec):
    data = H.synth("fastq", 3 << 20)
    a = codec.compress(data, 6)
    assert a == codec.compress(data, 6)
    # block-list path (the hook's) == bulk path, block by block
    blocks = [data[o : o + H.BLOCK] for o in range(0, len(data), H.BLOCK)]
    members, st = codec.compress_blocks(blocks[:7], 6)
    assert st == [0] * 7 and b"".join(members) == a[: sum(len(m) for m in members)]
    # sharding by contiguous block ranges (what 2/4/8 GPUs do) concatenates to the same stream
    import shard
    for world in (2, 4):
        parts = [codec.compress(data[slice(*shard.byte_range(len(data), H.BLOCK, r, world))], 6, eof=False) for r in range(world)]
        assert b"".join(parts) + H.EOF_BLOCK == a


@pytest.mark.parametrize("kind", ["fastq", "sam"])
@pytest.mark.parametrize("level", [1, 6, 12])
def test_inflate_reference_golden_streams_bit_exact(codec, kind, level):
    stream = open(os.path.join(H.GOLDEN, f"ref_{kind}_L{level}.bgz"), "rb").read()
    assert codec.inflate(stream + H.EOF_BLOCK) == H.synth(kind, 2 * H.BLOCK)


def test_inflate_large_reference_or_zlib_stream(codec):
    data = H.synth("fastq", 6 << 20) + H.lcg_noise(200000) + bytes(300000)
    if H.have_ref():
        stream, _, _ = H.Ref(6).compress_stream(data)
    else:
        stream = b"".join(H.zlib_member(data[o : o + H.BLOCK]) for o in range(0, len(data), H.BLOCK))
    out = codec.inflate(stream + H.EOF_BLOCK)
    assert out == data
    rc, oout, _ = H.oracle_decompress(stream)
    assert rc == 0 and oout == out


def test_inflate_zlib_members_all_block_types(codec):
    payload = H.synth("sam", 60000)
    stream = b""
    for level, strat in ((0, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_FIXED), (6, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_HUFFMAN_ONLY), (6, zlib.Z_RLE), (9, zlib.Z_FILTERED)):
        stream += H.zlib_member(payload, level, strat)
    # a member with several deflate blocks (sync flushes), and tiny members
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    raw = b"".join(co.compress(payload[o : o + 7000]) + co.flush(zlib.Z_FULL_FLUSH) for o in range(0, 56000, 7000)) + co.flush()
    stream += bytes.fromhex("1f8b08040000000000ff060042430200") + struct.pack("<H", len(raw) + 25) + raw + struct.pack("<II", zlib.crc32(payload[:56000]), 56000)
    stream += H.zlib_member(b"") + H.zlib_member(b"x") + H.EOF_BLOCK
    assert codec.inflate(stream) == payload * 6 + payload[:56000] + b"x"


def test_malformed_members_same_verdict_as_reference_decoder(codec):
    good = 0
    for c in MAL["cases"]:
        m = bytes.fromhex(c["hex"])
        try:
            out = codec.inflate(m)
            accepted = True
        except b200bgzf.B200BgzfError as e:
            assert e.code == -3
            accepted = False
        assert accepted == (c["ref_rc"] == 0), c["ref_rc"]
        if accepted:
            assert "%08x" % zlib.crc32(out) == c["ref_out_crc"]
            good += 1
    assert good > 5
    with pytest.raises(b200bgzf.B200BgzfError):
        codec.inflate(b"\x1f\x8b\x08\x00" + bytes(40))          # plain gzip is "not BGZF or corrupted" (7bgzf.c:313-316)


def test_reference_trees_malformed_vectors_are_rejected(codec):
    """the 151 malformed DEFLATE streams of lib/isa-l/igzip/inflate_std_vects.h (SURVEY 8c), one BGZF member each: same
    verdict as the reference decoder (it rejects every one), alone and in the middle of a batch of good members"""
    cases = json.load(open(os.path.join(H.GOLDEN, "isal_std_vects.json")))["cases"]
    assert len(cases) == 151
    good = codec.compress(H.synth("fastq", 3 * H.BLOCK), 6, eof=False)
    for c in cases:
        m = bytes.fromhex(c["hex"])
        for stream in (m, good + m + good):
            try:
                codec.inflate(stream)
                accepted = True
            except b200bgzf.B200BgzfError as e:
                assert e.code == -3
                accepted = False
            assert accepted == (c["ref_rc"] == 0), c["name"]
    assert codec.inflate(good + good) == H.synth("fastq", 3 * H.BLOCK) * 2     # the context is still healthy


def test_device_resident_api_roundtrip(codec):
    import torch
    data = H.synth("sam", 5 * H.BLOCK + 999)
    src = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    dst = torch.empty(codec.bound(len(data)), dtype=torch.uint8, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    n = codec.compress_device(src.data_ptr(), len(data), dst.data_ptr(), dst.numel(), 6, stream=s)
    comp = bytes(dst[:n].cpu().numpy())
    assert comp == H.emul_stream(data, 6)
    back = torch.empty(len(data) + 64, dtype=torch.uint8, device="cuda")
    m = codec.inflate_device(dst.data_ptr(), n, back.data_ptr(), back.numel(), stream=s)
    assert m == len(data) and bytes(back[:m].cpu().numpy()) == data
    # corrupt the BSIZE chain: must be reported as not-BGZF
    bad = dst.clone()
    bad[16] = (int(bad[16]) + 1) % 256
    with pytest.raises(b200bgzf.B200BgzfError):
        codec.inflate_device(bad.data_ptr(), n, back.data_ptr(), back.numel(), stream=s)


def test_device_index_ignores_signatures_inside_payloads(codec):
    """A stream whose payload holds BGZF headers (bgzip of a .bam / of a tar of .bgz files: incompressible, so it sits
    raw in stored members) must inflate on the device-resident path too: the member list is the BSIZE chain from offset 0
    (the reference's strictly sequential header walk, applet/7bgzf.c:306-330), not every signature hit."""
    import torch
    inner = codec.compress(H.synth("fastq", 40 * H.BLOCK + 77), 6)
    tiny = b"".join(codec.compress(b"x" * k, 6, eof=False) for k in range(1, 600))      # ~600 signatures within 20 KB
    tarlike = bytes(512) + inner + bytes(1024) + tiny + H.EOF_BLOCK * 3 + inner[:100000]
    s = torch.cuda.current_stream().cuda_stream
    for payload in (inner, tarlike):
        for level in (0, 1, 6):
            # level 0: stored members (what a compressor emits for data it cannot shrink): the embedded headers survive verbatim
            outer = codec.compress(payload, level) if level else b"".join(H.zlib_member(payload[o : o + 60000], 0) for o in range(0, len(payload), 60000)) + H.EOF_BLOCK
            nsig = outer.count(bytes.fromhex("1f8b08040000000000ff0600424302"))
            assert level or nsig > len(H.members(outer)) + 30
            assert codec.inflate(outer) == payload                                          # host header walk
            d = torch.frombuffer(bytearray(outer), dtype=torch.uint8).cuda()
            back = torch.empty(len(payload) + 64, dtype=torch.uint8, device="cuda")
            m = codec.inflate_device(d.data_ptr(), len(outer), back.data_ptr(), back.numel(), stream=s)
            assert m == len(payload) and bytes(back[:m].cpu().numpy()) == payload
            m = codec.inflate_device(d.data_ptr(), len(outer), back.data_ptr(), back.numel(), flags=b200bgzf.VERIFY, stream=s)
            assert m == len(payload)
            if H.have_ref():
                rc, out, _ = H.Ref(6).inflate_stream(outer)
                assert rc == 0 and out == payload
            # a stream that does not start with a member, or whose chain stops short of the end, is still refused
            for bad in (b"\0" + outer, outer + b"\0", outer[:-1]):
                d2 = torch.frombuffer(bytearray(bad), dtype=torch.uint8).cuda()
                with pytest.raises(b200bgzf.B200BgzfError) as e:
                    codec.inflate_device(d2.data_ptr(), len(bad), back.data_ptr(), back.numel(), stream=s)
                assert e.value.code == b200bgzf.E_FORMAT
    # three levels deep
    deep = codec.compress(codec.compress(codec.compress(H.synth("sam", 1 << 20), 6), 6), 6)
    d = torch.frombuffer(bytearray(deep), dtype=torch.uint8).cuda()
    back = torch.empty(len(deep) + 64, dtype=torch.uint8, device="cuda")
    m = codec.inflate_device(d.data_ptr(), len(deep), back.data_ptr(), back.numel(), stream=s)
    assert bytes(back[:m].cpu().numpy()) == codec.inflate(deep)


def test_near_optimal_block_list_calls_of_growing_size(codec):
    """hook lanes serve 1-block and 2-4-block calls alike: the four-candidate scratch of the near-optimal levels must be
    sized for the larger grid whichever comes first (ADVICE r1: out-of-bounds writes with 1 then 3 payloads at level 12)"""
    c2 = b200bgzf.Codec(0)
    try:
        data = H.synth("fastq", 4 * H.BLOCK)
        blocks = [data[o : o + H.BLOCK] for o in range(0, len(data), H.BLOCK)]
        for level in (12, 10):
            one, st = c2.compress_blocks(blocks[:1], level)
            assert st == [0]
            three, st = c2.compress_blocks(blocks[1:4], level)
            assert st == [0, 0, 0]
            four, st = c2.compress_blocks(blocks, level)
            assert st == [0] * 4 and four[:1] == one and four[1:] == three
            assert b"".join(four) + H.EOF_BLOCK == codec.compress(data, level)
            for m, b in zip(four, blocks):
                assert H.gunzip(m) == b
    finally:
        c2.close()


def test_multi_context_sharding_gives_the_single_gpu_stream(codec):
    """b200bgzf_multi_*: one host buffer fanned over G contexts as contiguous block ranges, shards joined at host-known
    offsets (SURVEY 8e).  On a one-GPU box the contexts share device 0; the stream must not depend on G."""
    data = H.synth("sam", 37 * H.BLOCK + 4321)
    want = codec.compress(data, 6)
    for devs in ([0], [0, 0], [0, 0, 0], [0] * 8):
        m = b200bgzf.MultiCodec(devs)
        try:
            assert m.count() == len(devs)
            assert m.compress(data, 6) == want
            assert m.compress(data[: 3 * H.BLOCK], 6) == codec.compress(data[: 3 * H.BLOCK], 6)    # fewer blocks than contexts
            assert m.compress(b"", 6) == H.EOF_BLOCK
            assert m.inflate(want) == data
            assert m.inflate(H.EOF_BLOCK) == b""
            with pytest.raises(b200bgzf.B200BgzfError):
                m.inflate(want[:-40] + b"garbage" + want[-33:])
        finally:
            m.close()


@pytest.mark.parametrize("level", [1, 6, 7, 9, 11])
def test_binary_corpus_three_byte_hash_window(codec, level):
    """an ELF binary (oracle/_ref/cielbox_ref): bytes of the CPU run of the same algorithm, decodes through the reference decoder,
    and — at the levels that hash three bytes on binary-looking blocks (6+) and at level 1 — within 3 % of the reference's size"""
    path = os.path.join(H.ROOT, "oracle", "_ref", "cielbox_ref")
    if not (H.have_ref() and os.path.exists(path)):
        pytest.skip("oracle/_ref not built")
    d = open(path, "rb").read()
    got = codec.compress(d, level)
    assert got == H.emul_stream(d, level)
    rc, out, _ = H.Ref(6).inflate_stream(got)
    assert rc == 0 and out == d and codec.inflate(got, flags=b200bgzf.VERIFY) == d
    _, ref_sizes, _ = H.Ref(level).compress_stream(d, keep=False, threads=os.cpu_count() or 1)
    assert len(got) - 28 <= 1.03 * sum(ref_sizes), (len(got), sum(ref_sizes))


def test_migz_members_on_the_same_kernel(codec):
    """SURVEY 8(f) rank 3, compress side: MiGz framing (gzip subfield "MZ" + u32 DEFLATE size, applet/7migz.c:224-233) around
    the same per-block DEFLATE data.  Decodes through the reference's own 7migz -d, gzip, and our inflate; the DEFLATE
    bytes of every member equal those of the BGZF member of the same payload."""
    data = H.synth("sam", 9 * 64512 + 777) + H.lcg_noise(3000) + bytes(5000)
    for level, blk in ((6, 64512), (1, 50000), (12, 64512)):
        mz = codec.compress(data, level, block_size=blk, flags=b200bgzf.FRAME_MIGZ)
        bz = codec.compress(data, level, block_size=blk, eof=False)
        assert H.gunzip(mz) == data and codec.inflate(mz) == data and codec.inflate(mz, flags=b200bgzf.VERIFY) == data
        off_m = off_b = 0
        nm = 0
        while off_m < len(mz):
            assert mz[off_m : off_m + 16] == bytes.fromhex("1f8b08040000000000ff08004d5a0400")
            csize = struct.unpack_from("<I", mz, off_m + 16)[0]
            bsize = struct.unpack_from("<H", bz, off_b + 16)[0] + 1
            assert mz[off_m + 20 : off_m + 20 + csize + 8] == bz[off_b + 18 : off_b + bsize]      # same DEFLATE data, CRC32 and ISIZE
            off_m += 20 + csize + 8
            off_b += bsize
            nm += 1
        assert off_m == len(mz) and off_b == len(bz) and nm == (len(data) + blk - 1) // blk
        if level == 6:
            H._emul().bgemul_set_header_bytes(20)
            try:
                assert mz == H.emul_stream(data, level, block=blk, eof=False)
            finally:
                H._emul().bgemul_set_header_bytes(18)
    ref_box = os.path.join(H.ROOT, "oracle", "_ref", "cielbox_ref")
    mz = codec.compress(data, 6, block_size=64512, flags=b200bgzf.FRAME_MIGZ)
    if os.path.exists(ref_box):
        r = subprocess.run([ref_box, "7migz", "-d"], input=mz, capture_output=True)
        assert r.returncode == 0 and r.stdout == data
    # the applet under its MiGz name: same stream; a member size the slots cannot hold is refused
    a = subprocess.run([b200bgzf.APPLET_PATH, "7migz", "-c", "-l6", "-b", "63"], input=data, capture_output=True)
    assert a.returncode == 0 and a.stdout == mz
    d = subprocess.run([b200bgzf.APPLET_PATH, "7migz", "-d"], input=a.stdout, capture_output=True)
    assert d.returncode == 0 and d.stdout == data
    # members of more than one slot (the reference's default: 512 KiB) are chains of pieces: tests/test_containers.py
    big = subprocess.run([b200bgzf.APPLET_PATH, "7migz", "-c", "-l6"], input=data, capture_output=True)
    assert big.returncode == 0 and big.stdout == codec.container(b200bgzf.CONTAINER_MIGZ, data, 6, 512)
    assert subprocess.run([b200bgzf.APPLET_PATH, "7migz", "-d"], input=big.stdout, capture_output=True).stdout == data
    if os.path.exists(ref_box):
        # ... and our inflate takes what the reference's 7migz writes (64 KiB members here; its default 512 KiB members too)
        for b in ("63", "512"):
            rr = subprocess.run([ref_box, "7migz", "-c", "-l6", "-b", b], input=data, capture_output=True)
            assert rr.returncode == 0 and codec.inflate(rr.stdout) == data
    m = b200bgzf.MultiCodec([0, 0, 0])
    try:
        assert m.compress(data, 6, block_size=64512, flags=b200bgzf.FRAME_MIGZ) == mz
    finally:
        m.close()


def test_verify_flag_checks_crc32_of_every_member(codec):
    """B200BGZF_VERIFY: CRC32 of the inflated payload against the trailer (the reference's decompress loop does not
    check it, applet/7bgzf.c:350-354): a flipped trailer byte is caught with the flag and ignored without."""
    import torch
    data = H.synth("fastq", 7 * H.BLOCK + 4321) + b"tail"
    if H.have_ref():
        ref_case = (H.Ref(6).compress_stream(data)[0] + H.EOF_BLOCK, data)
    else:                                                                     # the reference's committed two-block stream
        ref_case = (open(os.path.join(H.GOLDEN, "ref_fastq_L6.bgz"), "rb").read() + H.EOF_BLOCK, H.synth("fastq", 2 * H.BLOCK))
    for stream, data in ((codec.compress(data, 6), data), ref_case):
        assert codec.inflate(stream, flags=b200bgzf.VERIFY) == data          # intact: passes, host path
        mem = H.members(stream)
        off, size = mem[min(3, len(mem) - 2)][:2]                            # a data member (the reference's stream has two)
        for victim in (off + size - 8, off + size - 5):                      # first and last byte of the CRC32 field
            bad = bytearray(stream)
            bad[victim] ^= 0x40
            bad = bytes(bad)
            assert codec.inflate(bad) == data                                # like the reference: not checked
            with pytest.raises(b200bgzf.B200BgzfError) as e:
                codec.inflate(bad, flags=b200bgzf.VERIFY)
            assert e.value.code == b200bgzf.E_CRC
            d = torch.frombuffer(bytearray(bad), dtype=torch.uint8).cuda()
            back = torch.empty(len(data) + 64, dtype=torch.uint8, device="cuda")
            s = torch.cuda.current_stream().cuda_stream
            assert codec.inflate_device(d.data_ptr(), len(bad), back.data_ptr(), back.numel(), stream=s) == len(data)
            with pytest.raises(b200bgzf.B200BgzfError) as e:
                codec.inflate_device(d.data_ptr(), len(bad), back.data_ptr(), back.numel(), flags=b200bgzf.VERIFY, stream=s)
            assert e.value.code == b200bgzf.E_CRC
        # a payload byte changed by a literal flip (stream still decodes, same length): only the CRC can tell
    # odd sizes and unaligned output offsets: every member of a ragged stream verifies
    ragged = b"".join(codec.compress(H.synth("sam", n), 6, eof=False) for n in (1, 3, 17, 4097, 65280, 33333)) + H.EOF_BLOCK
    assert codec.inflate(ragged, flags=b200bgzf.VERIFY) == b"".join(H.synth("sam", n) for n in (1, 3, 17, 4097, 65280, 33333))


def test_inflate_other_block_gzip_flavours_like_the_reference_loop(codec):
    """the applet's decompress loop takes MiGz / mgzip members and optional header fields besides BGZF
    (applet/7bgzf.c:81-131); so do the host-buffer inflate and our applet; the fixtures are pinned by the reference
    applet in tests/test_abi.py"""
    from test_abi import _gz_member
    big, small = H.synth("sam", 200000), H.synth("fastq", 30000)
    parts = [(big, "migz", None), (small, "bgzf", b"reads.fq"), (big[:70001], "mgzip2", None), (small, "mgzip1", b"x"),
             (b"", "migz", None), (big, "migz", b"named")]
    stream = b"".join(_gz_member(d, f, name=n) for d, f, n in parts)
    want = b"".join(d for d, _, _ in parts)
    assert codec.inflate(stream) == want
    assert codec.inflate(stream, flags=b200bgzf.VERIFY) == want            # members <= 64 KiB are CRC-checked, larger ones pass
    bad = bytearray(stream)
    off = len(_gz_member(big, "migz"))                                      # the BGZF member's trailer CRC
    off += len(_gz_member(small, "bgzf", name=b"reads.fq")) - 8
    bad[off] ^= 1
    with pytest.raises(b200bgzf.B200BgzfError) as e:
        codec.inflate(bytes(bad), flags=b200bgzf.VERIFY)
    assert e.value.code == b200bgzf.E_CRC
    r = subprocess.run([b200bgzf.APPLET_PATH, "-d"], input=stream, capture_output=True)
    assert r.returncode == 0 and r.stdout == want
    if H.have_ref():
        # (without the empty member: the reference reads 64 header bytes at a time and gives up on members shorter than that)
        s2 = b"".join(_gz_member(d, f, name=n) for d, f, n in parts if d)
        rr = subprocess.run([os.path.join(H.ROOT, "oracle", "_ref", "7bgzf"), "-d"], input=s2, capture_output=True)
        assert rr.returncode == 0 and rr.stdout == want and codec.inflate(s2) == want
    # truncated last member / garbage: an error, not a hang or a partial success
    with pytest.raises(b200bgzf.B200BgzfError):
        codec.inflate(stream[:-3])
    with pytest.raises(b200bgzf.B200BgzfError):
        codec.inflate(stream + b"garbage after the last member")


HOOK_DRIVER = r"""
import ctypes, sys, threading
sys.path.insert(0, sys.argv[2]); sys.path.insert(0, sys.argv[3])
import helpers as H
hook = ctypes.CDLL(sys.argv[1])
hook.bgzf_compress.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_size_t), ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int]
data = H.synth("sam", 64 * H.BLOCK)
blocks = [data[o : o + H.BLOCK] for o in range(0, len(data), H.BLOCK)]
out = [None] * len(blocks)
def work(tid):
    dst = ctypes.create_string_buffer(65536)
    for i in range(tid, len(blocks), 8):
        n = ctypes.c_size_t(65536)
        assert hook.bgzf_compress(dst, ctypes.byref(n), blocks[i], len(blocks[i]), 9) == 0      # htslib's level is ignored
        out[i] = dst.raw[: n.value]
th = [threading.Thread(target=work, args=(t,)) for t in range(8)]
[t.start() for t in th]; [t.join() for t in th]
dst = ctypes.create_string_buffer(64)
n = ctypes.c_size_t(30); r1 = hook.bgzf_compress(dst, ctypes.byref(n), H.lcg_noise(1000), 1000, 6); k1 = n.value
n = ctypes.c_size_t(25); r2 = hook.bgzf_compress(dst, ctypes.byref(n), b"hello", 5, 6)
n = ctypes.c_size_t(64); r3 = hook.bgzf_compress(dst, ctypes.byref(n), b"", 0, 6); k3 = n.value
sys.stdout.buffer.write(b"".join(out))
sys.stderr.write("RC %d %d %d %d %d\n" % (r1, k1, r2, r3, k3))
"""


def test_hook_from_many_threads(codec, tmp_path):
    """LD_PRELOAD object: 8 concurrent callers (htslib's pool), BGZF_METHOD from the environment, reference return codes"""
    data = H.synth("sam", 64 * H.BLOCK)
    for method, level in (("libdeflate5", 5), ("LibDeflate", 6), (None, 6)):
        env = dict(os.environ)
        env.pop("BGZF_METHOD", None)
        if method:
            env["BGZF_METHOD"] = method
        r = subprocess.run([sys.executable, "-c", HOOK_DRIVER, b200bgzf.HOOK_PATH, os.path.join(H.ROOT, "tests"), os.path.join(H.ROOT, "7bgzf_b200")],
                           capture_output=True, env=env)
        assert r.returncode == 0, r.stderr.decode()
        assert r.stdout + H.EOF_BLOCK == codec.compress(data, level)
        tail = [l for l in r.stderr.decode().splitlines() if l.startswith("RC ")][-1].split()[1:]
        assert tail == ["1", "30", "-1", "0", "28"]           # does-not-fit -> 1 (*dlen untouched); cap < 26 -> -1; slen 0 -> EOF block
        assert "libdeflate_deflate 1" in r.stderr.decode()     # the reference's stderr line for the does-not-fit case
    # the combiner path (what >36 concurrent callers get: payloads pooled into batches by one dispatcher thread): same bytes, same codes
    for method, level in (("libdeflate6", 6), ("libdeflate10", 10)):
        env = dict(os.environ, BGZF_METHOD=method, B200BGZF_HOOK_BATCH="1")
        r = subprocess.run([sys.executable, "-c", HOOK_DRIVER, b200bgzf.HOOK_PATH, os.path.join(H.ROOT, "tests"), os.path.join(H.ROOT, "7bgzf_b200")],
                           capture_output=True, env=env)
        assert r.returncode == 0, r.stderr.decode()
        assert r.stdout + H.EOF_BLOCK == codec.compress(data, level)
        tail = [l for l in r.stderr.decode().splitlines() if l.startswith("RC ")][-1].split()[1:]
        assert tail == ["1", "30", "-1", "0", "28"]
    env = dict(os.environ, BGZF_METHOD="libdeflate13")
    r = subprocess.run([sys.executable, "-c", HOOK_DRIVER, b200bgzf.HOOK_PATH, os.path.join(H.ROOT, "tests"), os.path.join(H.ROOT, "7bgzf_b200")],
                       capture_output=True, env=env)
    assert r.returncode != 0                                   # out-of-range level: every call fails with -1, nothing crashes


SPLIT_DRIVER = r"""
import sys
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2])
import helpers as H, b200bgzf
c = b200bgzf.Codec(0)
fq, sam = H.synth("fastq", 3 * H.BLOCK), H.synth("sam", 0x10000)
cases = [fq[:H.BLOCK], fq[H.BLOCK:2 * H.BLOCK], sam, sam[:8192], sam[:8191], sam[:20001], H.lcg_noise(H.BLOCK), bytes(H.BLOCK),
         H.acgt(H.BLOCK), H.bamlike(H.BLOCK), fq[:1025], fq[:4 * 1024 + 1]]
for level in (1, 4, 6, 9, 10):
    for pl in cases:
        got, st = c.compress_blocks([pl], level)
        assert st == [0], (level, len(pl), st)
        sys.stdout.buffer.write(got[0])
"""


def test_one_member_calls_on_a_cluster_give_the_same_bytes(codec):
    """the hook's one-block path lets a cluster of 2/4/8 CTAs share the search of the block: every size must give the
    bytes of the one-CTA kernel (= the emulator's), for all classes that split (greedy/lazy) and one that does not (10)"""
    fq, sam = H.synth("fastq", 3 * H.BLOCK), H.synth("sam", 0x10000)
    cases = [fq[:H.BLOCK], fq[H.BLOCK:2 * H.BLOCK], sam, sam[:8192], sam[:8191], sam[:20001], H.lcg_noise(H.BLOCK), bytes(H.BLOCK),
             H.acgt(H.BLOCK), H.bamlike(H.BLOCK), fq[:1025], fq[:4 * 1024 + 1]]
    want = b"".join(codec.compress(pl, level, 0x10000, eof=False) for level in (1, 4, 6, 9, 10) for pl in cases)
    e0 = H.emul_block(cases[0], 1)[1]
    assert want[: len(e0)] == e0
    for split in ("1", "2", "4", "8", ""):
        env = dict(os.environ, B200BGZF_SPLIT=split)
        r = subprocess.run([sys.executable, "-c", SPLIT_DRIVER, os.path.join(H.ROOT, "tests"), os.path.join(H.ROOT, "7bgzf_b200")],
                           capture_output=True, env=env)
        assert r.returncode == 0, r.stderr.decode()
        assert r.stdout == want, split


def test_applet_roundtrip_and_stderr_contract():
    data = H.synth("fastq", 3 << 20)
    r = subprocess.run([b200bgzf.APPLET_PATH, "-c", "-l6", "-@", "4"], input=data, capture_output=True)
    assert r.returncode == 0
    err = r.stderr.decode()
    assert "compression level = 6 (libdeflate)" in err and " done." in err and "ellapsed time:" in err
    assert r.stdout == H.emul_stream(data, 6)
    d = subprocess.run([b200bgzf.APPLET_PATH, "-d"], input=r.stdout, capture_output=True)
    assert d.returncode == 0 and d.stdout == data
    if os.path.exists(H.REF_7BGZF):
        ref = subprocess.run([H.REF_7BGZF, "-c", "-l6", "-@", "4"], input=data, capture_output=True)
        d2 = subprocess.run([b200bgzf.APPLET_PATH, "-d"], input=ref.stdout, capture_output=True)
        assert d2.returncode == 0 and d2.stdout == data            # our applet inflates the reference applet's stream
        assert len(r.stdout) <= 1.03 * len(ref.stdout)
    bad = subprocess.run([b200bgzf.APPLET_PATH, "-d"], input=b"this is not bgzf at all, not even close........", capture_output=True)
    assert bad.returncode != 0 and b"not BGZF or corrupted" in bad.stderr
    # block size rule of the reference (7bgzf.c:141-147): one thread (the default) cuts 0x10000-byte blocks, -@N 0xff00-byte ones
    r1 = subprocess.run([b200bgzf.APPLET_PATH, "-c", "-l6"], input=data, capture_output=True)
    assert r1.returncode == 0 and r1.stdout == H.emul_stream(data, 6, 0x10000)
    assert [m[2] for m in H.members(r1.stdout)[:2]] == [0x10000, 0x10000]
    if os.path.exists(H.REF_7BGZF):
        ref1 = subprocess.run([H.REF_7BGZF, "-c", "-l6"], input=data, capture_output=True)
        assert [m[2] for m in H.members(ref1.stdout)[:-1]] == [m[2] for m in H.members(r1.stdout)[:-1]]   # same block boundaries
        assert len(r1.stdout) <= 1.03 * len(ref1.stdout)
    # ... and a 0x10000-byte block that does not compress cannot fit a member: the slot is redone in 0xff00-byte blocks
    noisy = H.lcg_noise(3 * 0x10000 + 777) + data[:100000]
    rn = subprocess.run([b200bgzf.APPLET_PATH, "-c", "-l6"], input=noisy, capture_output=True)
    assert rn.returncode == 0 and H.gunzip(rn.stdout) == noisy and rn.stdout == H.emul_stream(noisy, 6)


def test_member_offsets_and_gzi_index(codec, tmp_path):
    """SURVEY §8(f) rank 2: the member offsets of the device scan, as an ABI output and as the applet's --gzi file;
    checked against a header walk of the stream, and used for random access"""
    data = H.synth("fastq", 5 * 1024 * 1024 + 321) + H.lcg_noise(70000) + bytes(100000)
    for blk in (0xFF00, 0x10000 - 64):
        stream, offs = codec.compress_indexed(data, 6, blk)
        assert stream == codec.compress(data, 6, blk)
        mem = H.members(stream)
        assert offs == [m[0] for m in mem[:-1]]
        nb = len(offs)
        gzi = b200bgzf.gzi_format(offs, [b * blk for b in range(nb)])
        assert gzi == H.gzi_of(stream)
        # random access through the index: one member inflated on its own is the payload at its uncompressed address
        for b in (0, 1, nb // 2, nb - 1):
            one = stream[offs[b] : offs[b] + mem[b][1]]
            assert codec.inflate(one) == data[b * blk : (b + 1) * blk]
    # more blocks than one pipelined batch (512) and than one lane rotation
    big = H.synth("sam", 48 << 20)
    stream, offs = codec.compress_indexed(big, 1)
    assert offs == [m[0] for m in H.members(stream)[:-1]] and H.gunzip(stream) == big
    assert codec.compress_indexed(b"", 6) == (b200bgzf.EOF_BLOCK, [])
    # the applet writes the same index (-@4: 0xff00-byte blocks; default: 0x10000, with a slot redone at 0xff00)
    for args, src in ((["-@", "4"], data), ([], data), ([], big[: 40 << 20])):
        path = tmp_path / "x.gzi"
        r = subprocess.run([b200bgzf.APPLET_PATH, "-c", "-l6", "--gzi=%s" % path] + args, input=src, capture_output=True)
        assert r.returncode == 0, r.stderr
        assert r.stdout == subprocess.run([b200bgzf.APPLET_PATH, "-c", "-l6"] + args, input=src, capture_output=True).stdout
        assert path.read_bytes() == H.gzi_of(r.stdout)
        os.unlink(path)


def test_full_size_properties_1gib(codec):
    """BASELINE configs[0]/[1] size: 1 GiB FASTQ-like.  Size-independent properties: round trip through our
    inflate, ISIZE sum, per-block CRC32 against zlib on a sample, combined CRC of the whole payload."""
    import numpy as np
    import torch
    n = 1 << 30
    host = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    H._gen().b200gen_fill(0, 1, host.data_ptr(), n)
    out = torch.empty(codec.bound(n), dtype=torch.uint8, pin_memory=True)
    clen = codec.compress_into(host.data_ptr(), n, out.data_ptr(), out.numel(), 6)
    assert 0.20 * n < clen < 0.26 * n                                   # reference libdeflate6 ratio on this corpus: 0.2406
    view = out.numpy()[:clen]
    back = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    m = codec.inflate_into(out.data_ptr(), clen, back.data_ptr(), n)
    assert m == n and torch.equal(back, host)
    # trailer fields of a sample of members + checksum of checksums
    raw = view.tobytes()
    mem = H.members(raw)
    assert len(mem) == (n + H.BLOCK - 1) // H.BLOCK + 1 and sum(x[2] for x in mem) == n
    hb = host.numpy()
    crc_all = 0
    o = H.oracle()
    for i, (off, size, isize, crc) in enumerate(mem[:-1]):
        if i % 257 == 0:
            assert crc == zlib.crc32(hb[i * H.BLOCK : i * H.BLOCK + isize].tobytes())
        crc_all = o.oracle_crc32_combine(crc_all, crc, isize)
    assert crc_all == zlib.crc32(hb)
    if H.have_ref():
        # the whole 1 GiB stream through the reference's own libdeflate decoder (all host threads), bit-exact
        o2 = H.oracle()
        n_out, rc = ctypes.c_size_t(), ctypes.c_int()
        back.zero_()
        t = o2.refh_inflate(H.Ref(6).h, out.data_ptr(), clen, os.cpu_count() or 1, back.data_ptr(), n, ctypes.byref(n_out), ctypes.byref(rc))
        assert t >= 0 and rc.value == 0 and n_out.value == n and torch.equal(back, host)


def test_full_size_near_optimal_256mib_through_reference_decoder(codec):
    """BASELINE config 4's class at 256 MiB: the level-12 stream decodes bit-exactly through the reference's decoder and
    stays within 3 % of the reference's level-12 size (the reference compresses a 4 MiB sample: ~1 MB/s per core)"""
    import torch
    if not H.have_ref():
        pytest.skip("oracle/_ref not built")
    n = 256 << 20
    host = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    H._gen().b200gen_fill(0, 1, host.data_ptr(), n)
    out = torch.empty(codec.bound(n), dtype=torch.uint8, pin_memory=True)
    clen = codec.compress_into(host.data_ptr(), n, out.data_ptr(), out.numel(), 12)
    back = torch.zeros(n, dtype=torch.uint8, pin_memory=True)
    n_out, rc = ctypes.c_size_t(), ctypes.c_int()
    t = H.oracle().refh_inflate(H.Ref(12).h, out.data_ptr(), clen, os.cpu_count() or 1, back.data_ptr(), n, ctypes.byref(n_out), ctypes.byref(rc))
    assert t >= 0 and rc.value == 0 and n_out.value == n and torch.equal(back, host)
    sample = 64 * H.BLOCK
    _, ref_sizes, _ = H.Ref(12).compress_stream(ctypes.string_at(host.data_ptr(), sample), keep=False, threads=os.cpu_count() or 1)
    ours = sum(m[1] for m in H.members(ctypes.string_at(out.data_ptr(), clen))[: sample // H.BLOCK])
    assert ours <= 1.03 * sum(ref_sizes), (ours, sum(ref_sizes))


def test_checked_build_bounds_asserts_stay_silent():
    """compute-sanitizer is not available on the GPU pool; instead the indices the kernels compute (search bitmaps, candidate
    queues, position rings, scratch words, chunk order, compaction offsets) are asserted in a separate build (`make checked`,
    -DBG_CHECK).  The parity tests that exercise those paths are run once more against that library: an assert that fires
    traps, the launch fails, and so does the test."""
    lib = os.path.join(H.ROOT, "build", "checked", "lib7bgzf_b200.so")
    if not os.path.exists(lib):
        pytest.skip("build/checked missing: make checked")
    env = dict(os.environ, B200BGZF_LIB_PATH=lib)
    sel = "edge_inputs or whole_stream or binary_corpus or near_optimal_block or migz or multi_context or odd_block_sizes or bam_like or device_index"
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(H.ROOT, "tests", "test_gpu.py"), "-q", "-x", "-m", "gpu", "-k", sel,
                        "-p", "no:cacheprovider"], capture_output=True, text=True, env=env, cwd=H.ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "BG_ASSERT failed" not in r.stdout + r.stderr
    assert " passed" in r.stdout
