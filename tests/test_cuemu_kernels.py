"""CPU: the CUDA kernel SOURCES compiled for the host through tests/cuemu/cuemu.h (a fiber-per-thread emulation of the
warp-synchronous subset they use) against the oracle.  This is a logic check of the kernel code on a machine without a GPU --
not a CPU path of the product (libb200z.so is nvcc-only and fails without a device) and no substitute for the `-m gpu` parity
tests: it cannot see timing, memory-model races between warps or anything about the hardware.

  * zstd_enc_find_kernel / zstd_enc_dp_kernel (stage F / stage G: the level-3-class finder and parse) were developed against it
    (named barriers and shared-memory atomicMax included).
  * lzma2_cand_kernel / lzma2_parse_kernel (stage C / stage P of the price-based LZMA2 parse) and zstd_enc_parse_kernel
    (stage Z, the price-based Zstandard parse) were developed against it."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import helpers as H

HERE = os.path.dirname(os.path.abspath(__file__))
OPT = 0x10


@pytest.fixture(scope="module")
def emu():
    E = H.cuemu_library()
    vp, u32, u64 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64
    E.emu_zstd_enc_match.restype = u64; E.emu_zstd_enc_match.argtypes = [vp, u64, u32, u32, u32, u32, u32, vp, vp, vp, vp]
    E.emu_zstd_enc_find.restype = u64; E.emu_zstd_enc_find.argtypes = [vp, u64, u32, u32, u32, u32, u32, vp]
    E.emu_zstd_enc_find_long.restype = u64; E.emu_zstd_enc_find_long.argtypes = [vp, u64, u32, u32, u32, u32, u32, vp]
    E.emu_lzma2_cand.restype = u64; E.emu_lzma2_cand.argtypes = [vp, u64, u32, u32, u32, vp]
    E.emu_lzma2_parse.restype = u64; E.emu_lzma2_parse.argtypes = [vp, u64, u32, u32, vp, vp, vp]
    E.emu_zstd_enc_parse.restype = u64; E.emu_zstd_enc_parse.argtypes = [vp, u64, u32, u32, vp, vp, vp, vp, vp]
    E.emu_zstd_enc_entropy.restype = u64; E.emu_zstd_enc_entropy.argtypes = [vp, u64, u32, u32, vp, vp, vp, vp, vp, vp, u32]
    E.emu_slot_bytes.restype = u32
    i64 = ctypes.c_int64
    E.emu_lzma2_range_and_assemble.restype = i64; E.emu_lzma2_range_and_assemble.argtypes = [vp, u64, u32, u32, vp, vp, vp, u64, ctypes.c_int]
    E.emu_zstd_enc_assemble.restype = i64; E.emu_zstd_enc_assemble.argtypes = [vp, u64, u32, u32, vp, vp, u32, vp, u64]
    E.emu_zstd_decode.restype = i64; E.emu_zstd_decode.argtypes = [vp, u64, vp, u64]
    E.emu_lzma2_decode.restype = i64; E.emu_lzma2_decode.argtypes = [vp, u64, u32, vp, u64, ctypes.c_int]
    E.emu_zstd_decode_jump.restype = i64; E.emu_zstd_decode_jump.argtypes = [vp, u64, vp, u64, u32, vp]
    return E


def _mixed(pkg, n_text):
    return (pkg.corpus.g2(n_text).tobytes() + bytes(5000) + pkg.corpus.entropy_class(3, 70_000).tobytes() + b"ab" * 3000
            + pkg.corpus.entropy_class(1, 20_000).tobytes() + pkg.corpus.entropy_class(2, 30_000).tobytes())


@pytest.mark.parametrize("fl,cl,ctas", [(17, 7, 2), (18, 5, 1), (17, 8, 3), (19, 6, 1)])
def test_emulated_stage_f_equals_the_oracle(pkg, emu, fl, cl, ctas):
    """candidate words of zstd_enc_find_kernel == b2zo_zstd_candidates for every chunk size the kernel is instantiated for"""
    data = _mixed(pkg, 150_000) + b"xyzw" * 700 + bytes(3); n = len(data)
    src = np.frombuffer(data + bytes(64), dtype=np.uint8)
    want = H.oracle_candidates(data, frameLog=fl, windowLog=fl, chunkLog=cl)
    got = np.full(((n + (1 << fl) - 1) >> fl << fl) + 16, 0xCDCDCDCD, dtype=np.uint32)
    emu.emu_zstd_enc_find(src.ctypes.data, n, fl, fl, cl, 1, ctas, got.ctypes.data)         # (returns the count of warp collectives: stage F has none)
    assert np.array_equal(got[:n], want)
    assert int((want != 0).sum()) > n // 4


@pytest.mark.parametrize("level,flag", [(1, 0x40), (6, 0x80)])
def test_emulated_stage_f_level_ladder(pkg, emu, level, flag):
    """the other rungs of stage F's ladder: levels 1-2 keep only the short table (in the long table's room), levels 5-7 let a position
    see the lower lanes of its own step (__match_any_sync) -- kernel == oracle for both"""
    data = _mixed(pkg, 120_000) + b"0123456789" * 2000; n = len(data); fl = 17
    src = np.frombuffer(data + bytes(64), dtype=np.uint8)
    p = H.EncParams(); H.oracle().b2zo_enc_default_params(ctypes.byref(p), level)
    assert p.flags & 0xC0 == flag
    want = H.oracle_candidates(data, frameLog=fl, windowLog=fl, flags=p.flags, hashLogS=p.hashLogS)
    got = np.full(((n + (1 << fl) - 1) >> fl << fl) + 16, 0xCDCDCDCD, dtype=np.uint32)
    emu.emu_zstd_enc_find(src.ctypes.data, n, fl, fl, 7, p.flags, 2, got.ctypes.data)
    assert np.array_equal(got[:n], want)
    base = H.oracle_candidates(data, frameLog=fl, windowLog=fl)
    assert not np.array_equal(base, want)


@pytest.mark.parametrize("fl,wl,rl,ll,ctas", [(20, 19, 17, 12, 2), (19, 19, 17, 10, 1), (21, 18, 17, 11, 3)])
def test_emulated_long_mode_candidates_equal_the_oracle(pkg, emu, fl, wl, rl, ll, ctas):
    """long mode: stage F per region + the two passes of zstd_enc_ldm_kernel == b2zo_zstd_candidates (regions, stage L's samples and
    epoch tables, the window, the walk back to the start of the agreement, the keep-the-nearer rule), on data with copies planted
    all over the frame, some mutated"""
    data = H.far_copies(pkg, (5 << 18) + 12345, every=1 << 17, span=(20_000, 60_000), seed=fl)
    n = len(data)
    src = np.frombuffer(data + bytes(64), dtype=np.uint8)
    want = H.oracle_candidates(data, frameLog=fl, windowLog=wl, regionLog=rl, ldmLog=ll)
    plain = H.oracle_candidates(data, frameLog=fl, windowLog=wl, regionLog=rl, ldmLog=0)
    off = want >> 5
    assert int((off >= (1 << rl)).sum()) > 50 and not np.array_equal(want, plain)          # stage L did find matches further back than a region
    assert int(off.max()) < (1 << wl)                                                        # ... and none beyond the window
    if fl > wl:
        assert int((off > (1 << (wl - 1))).sum()) > 5                                         # found through the table of an earlier epoch
    got = np.full(((n + (1 << fl) - 1) >> fl << fl) + 16, 0xCDCDCDCD, dtype=np.uint32)
    emu.emu_zstd_enc_find_long(src.ctypes.data, n, fl, wl, rl, ll, ctas, got.ctypes.data)
    assert np.array_equal(got[:n], want)


def test_emulated_stage_f_g_edge_inputs(pkg, emu):
    """tiny, ragged and degenerate frames through stage F + stage G: fewer bytes than a hash, one repeated byte (the RLE-block
    sequence), a block that ends one byte into a segment, long matches that stage G extends past B2Z_CAP"""
    cases = [b"a", b"ab", b"abcdefg", b"abcabcabcabc", bytes(70_000), b"\x07" * 131072 + b"\x07", pkg.corpus.g2(131073).tobytes(), b"\x01" * 33,
             pkg.corpus.g2(40_000).tobytes() * 3, pkg.corpus.g2(4097).tobytes(), (b"0123456789abcdef" * 300 + b"Z") * 9]
    for data in cases:
        n = len(data); fl = 17
        src = np.frombuffer(data + bytes(64), dtype=np.uint8)
        nblk = (n + 131071) // 131072
        seqs, nseq, lits, nlit = H.oracle_find_sequences(data, frameLog=fl, windowLog=fl)
        s2 = np.zeros(nblk * H.MAXSEQ, dtype=np.uint64); ns2 = np.zeros(nblk, dtype=np.uint32); nl2 = np.zeros(nblk, dtype=np.uint32); l2 = np.zeros(nblk * 131072 + 64, dtype=np.uint8)
        emu.emu_zstd_enc_match(src.ctypes.data, n, fl, fl, 7, 1, 2, s2.ctypes.data, ns2.ctypes.data, l2.ctypes.data, nl2.ctypes.data)
        assert np.array_equal(nseq, ns2) and np.array_equal(nlit, nl2), n
        for b in range(nblk):
            assert np.array_equal(seqs[b * H.MAXSEQ:b * H.MAXSEQ + nseq[b]], s2[b * H.MAXSEQ:b * H.MAXSEQ + nseq[b]]), (n, b)
            assert np.array_equal(lits[b * 131072:b * 131072 + nlit[b]], l2[b * 131072:b * 131072 + nlit[b]]), (n, b)


def test_emulated_stage_m_equals_the_oracle(pkg, emu):
    data = _mixed(pkg, 200_000); n = len(data)
    src = np.frombuffer(data + bytes(64), dtype=np.uint8)
    nblk = (n + 131071) // 131072
    for fl, warps in ((17, 2), (18, 1)):
        seqs, nseq, lits, nlit = H.oracle_find_sequences(data, frameLog=fl, windowLog=fl)
        s2 = np.zeros(nblk * H.MAXSEQ, dtype=np.uint64); ns2 = np.zeros(nblk, dtype=np.uint32); nl2 = np.zeros(nblk, dtype=np.uint32); l2 = np.zeros(n + 64, dtype=np.uint8)
        assert emu.emu_zstd_enc_match(src.ctypes.data, n, fl, fl, 7, 1 | (2 << 8), warps, s2.ctypes.data, ns2.ctypes.data, l2.ctypes.data, nl2.ctypes.data) > 0
        assert np.array_equal(nseq, ns2) and np.array_equal(nlit, nl2)
        for b in range(nblk):
            assert np.array_equal(seqs[b * H.MAXSEQ:b * H.MAXSEQ + nseq[b]], s2[b * H.MAXSEQ:b * H.MAXSEQ + nseq[b]]), b
            assert np.array_equal(lits[b * 131072:b * 131072 + nlit[b]], l2[b * 131072:b * 131072 + nlit[b]]), b


def _oracle_taps(data, fl, flags):
    O = H.oracle()
    O.b2zo_lzma2_candidates.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p]
    O.b2zo_lzma2_parse_frame.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.POINTER(H.EncParams)] + [ctypes.c_void_p] * 3
    n = len(data); F = 1 << fl; bpf = F >> 17; nfr = (n + F - 1) // F
    src = np.frombuffer(data, dtype=np.uint8)
    cand = np.zeros(nfr * F * 4, dtype=np.uint32); seqs = np.zeros(nfr * bpf * H.MAXSEQ, dtype=np.uint64); nseq = np.zeros(nfr * bpf, dtype=np.uint32)
    p = H.enc_params(frameLog=fl, windowLog=fl, flags=flags)
    for f in range(nfr):
        f0 = f * F; fn = min(F, n - f0)
        O.b2zo_lzma2_candidates(src.ctypes.data + f0, fn, fl, cand.ctypes.data + f0 * 16)
        O.b2zo_lzma2_parse_frame(src.ctypes.data + f0, fn, ctypes.byref(p), cand.ctypes.data + f0 * 16, seqs.ctypes.data + f * bpf * H.MAXSEQ * 8, nseq.ctypes.data + f * bpf * 4)
    return cand, seqs, nseq


@pytest.mark.parametrize("fl,sl,warps", [(18, 1, 2), (17, 0, 3), (19, 2, 1)])
def test_emulated_stage_c_and_p_equal_the_oracle(pkg, emu, fl, sl, warps):
    data = _mixed(pkg, 150_000); n = len(data)
    flags = 1 | (sl << 8) | OPT
    src = np.frombuffer(data + bytes(64), dtype=np.uint8)
    candO, seqO, nsO = _oracle_taps(data, fl, flags)
    candE = np.zeros_like(candO)
    assert emu.emu_lzma2_cand(src.ctypes.data, n, fl, flags, warps, candE.ctypes.data) > 0
    assert np.array_equal(candE[:n * 4], candO[:n * 4])
    seqE = np.zeros_like(seqO); nsE = np.full_like(nsO, 0xFFFFFFFF)
    assert emu.emu_lzma2_parse(src.ctypes.data, n, fl, flags, candE.ctypes.data, seqE.ctypes.data, nsE.ctypes.data) > 0
    assert np.array_equal(nsE, nsO) and int(nsO.sum()) > 10_000
    for b in range(len(nsO)):
        assert np.array_equal(seqE[b * H.MAXSEQ:b * H.MAXSEQ + nsO[b]], seqO[b * H.MAXSEQ:b * H.MAXSEQ + nsO[b]]), b


def test_emulated_parse_edge_inputs(pkg, emu):
    """tiny, ragged and degenerate frames: one byte, shorter than any key, all zeros (every window ends in a long match),
    a frame that ends one byte into a block"""
    cases = [b"a", b"ab", b"abcabcabcabc", bytes(70_000), pkg.corpus.g2(131073).tobytes(), b"\x01" * 33, pkg.corpus.g2(40_000).tobytes() * 3]
    for data in cases:
        n = len(data); fl = 17; flags = 1 | OPT
        src = np.frombuffer(data + bytes(64), dtype=np.uint8)
        candO, seqO, nsO = _oracle_taps(data, fl, flags)
        candE = np.zeros_like(candO); seqE = np.zeros_like(seqO); nsE = np.full_like(nsO, 0xFFFFFFFF)
        emu.emu_lzma2_cand(src.ctypes.data, n, fl, flags, 2, candE.ctypes.data)
        assert np.array_equal(candE[:n * 4], candO[:n * 4]), n
        emu.emu_lzma2_parse(src.ctypes.data, n, fl, flags, candE.ctypes.data, seqE.ctypes.data, nsE.ctypes.data)
        nb = (n + 131071) // 131072
        assert np.array_equal(nsE[:nb], nsO[:nb]), n
        for b in range(nb):
            assert np.array_equal(seqE[b * H.MAXSEQ:b * H.MAXSEQ + nsO[b]], seqO[b * H.MAXSEQ:b * H.MAXSEQ + nsO[b]]), (n, b)


ZOPT = 0x20


@pytest.mark.parametrize("fl", [17, 18])
def test_emulated_stage_z_equals_the_oracle(pkg, emu, fl):
    data = _mixed(pkg, 200_000) + bytes(150_000); n = len(data)
    flags = 1 | ZOPT
    src = np.frombuffer(data + bytes(64), dtype=np.uint8)
    seqO, nsO, litO, nlO = H.oracle_find_sequences(data, frameLog=fl, windowLog=fl, flags=flags)
    F = 1 << fl; nfr = (n + F - 1) // F
    cand = np.zeros(nfr * F * 4, dtype=np.uint32)
    emu.emu_lzma2_cand(src.ctypes.data, n, fl, flags, 2, cand.ctypes.data)
    seqE = np.zeros_like(seqO); nsE = np.full_like(nsO, 0xFFFFFFFF); nlE = np.full_like(nlO, 0xFFFFFFFF); litE = np.zeros(n + 64, dtype=np.uint8)
    assert emu.emu_zstd_enc_parse(src.ctypes.data, n, fl, flags, cand.ctypes.data, seqE.ctypes.data, nsE.ctypes.data, litE.ctypes.data, nlE.ctypes.data) > 0
    assert np.array_equal(nsE, nsO) and np.array_equal(nlE, nlO) and int(nsO.sum()) > 10_000
    for b in range(len(nsO)):
        assert np.array_equal(seqE[b * H.MAXSEQ:b * H.MAXSEQ + nsO[b]], seqO[b * H.MAXSEQ:b * H.MAXSEQ + nsO[b]]), b
        assert np.array_equal(litE[b * 131072:b * 131072 + nlO[b]], litO[b * 131072:b * 131072 + nlO[b]]), b


def test_emulated_stage_z_edge_inputs(pkg, emu):
    cases = [b"a", b"ab", b"abcabcabcabc", bytes(70_000), pkg.corpus.g2(131073).tobytes(), b"\x01" * 33, pkg.corpus.g2(40_000).tobytes() * 3,
             pkg.corpus.entropy_class(1, 50_000).tobytes()]
    for data in cases:
        n = len(data); fl = 17; flags = 1 | ZOPT
        src = np.frombuffer(data + bytes(64), dtype=np.uint8)
        seqO, nsO, litO, nlO = H.oracle_find_sequences(data, frameLog=fl, windowLog=fl, flags=flags)
        nfr = (n + (1 << fl) - 1) >> fl
        cand = np.zeros(nfr * (1 << fl) * 4, dtype=np.uint32)
        emu.emu_lzma2_cand(src.ctypes.data, n, fl, flags, 1, cand.ctypes.data)
        seqE = np.zeros_like(seqO); nsE = np.full_like(nsO, 0xFFFFFFFF); nlE = np.full_like(nlO, 0xFFFFFFFF); litE = np.zeros(n + 64, dtype=np.uint8)
        emu.emu_zstd_enc_parse(src.ctypes.data, n, fl, flags, cand.ctypes.data, seqE.ctypes.data, nsE.ctypes.data, litE.ctypes.data, nlE.ctypes.data)
        assert np.array_equal(nsE, nsO) and np.array_equal(nlE, nlO), n
        for b in range(len(nsO)):
            assert np.array_equal(seqE[b * H.MAXSEQ:b * H.MAXSEQ + nsO[b]], seqO[b * H.MAXSEQ:b * H.MAXSEQ + nsO[b]]), (n, b)
            assert np.array_equal(litE[b * 131072:b * 131072 + nlO[b]], litO[b * 131072:b * 131072 + nlO[b]]), (n, b)


@pytest.mark.parametrize("fl,flags", [(18, 1 | ZOPT), (17, 1 | ZOPT), (18, 1)])
def test_emulated_stage_e_codes_stage_z_sequences_like_the_oracle(pkg, emu, fl, flags):
    """stage E (zstd_enc_entropy_kernel) is GPU-verified on stage M's sequences; stage Z hands it shapes stage M never produces
    (length-3 matches, tiny offsets, up to 32 768 sequences per block): its emulated output on those must be the oracle's blocks."""
    import struct
    data = (pkg.corpus.g2(600_000).tobytes() + bytes(5000) + pkg.corpus.entropy_class(3, 100_000).tobytes() + b"ab" * 3000
            + pkg.corpus.entropy_class(1, 140_000).tobytes() + bytes(200_000) + pkg.corpus.entropy_class(2, 100_000).tobytes())
    n = len(data); F = 1 << fl; SLOT = emu.emu_slot_bytes()
    src = np.frombuffer(data + bytes(64), dtype=np.uint8)
    seqO, nsO, litO, nlO = H.oracle_find_sequences(data, frameLog=fl, windowLog=fl, flags=flags)
    nblk = len(nsO)
    lits = np.zeros(n + 64, dtype=np.uint8); lits[:n] = litO
    slots = np.zeros(nblk * SLOT, dtype=np.uint8); ssz = np.zeros(nblk, dtype=np.uint32)
    assert emu.emu_zstd_enc_entropy(src.ctypes.data, n, fl, flags, seqO.ctypes.data, nsO.ctypes.data, lits.ctypes.data, nlO.ctypes.data,
                                    slots.ctypes.data, ssz.ctypes.data, nblk) > 0
    comp = H.oracle_compress(data, frameLog=fl, windowLog=fl, flags=flags)
    ip = 0; blk = 0
    for f0 in range(0, n, F):                                       # the oracle's frames: [12-byte size hint][10-byte header, blocks ...]
        assert comp[ip:ip + 4] == b"\x50\x2a\x4d\x18"
        fsize = struct.unpack("<I", comp[ip + 8:ip + 12])[0]; ip += 12
        body = comp[ip + 10:ip + fsize]; ip += fsize
        nb = (min(F, n - f0) + 131071) // 131072
        mine = b"".join(slots[b * SLOT:b * SLOT + ssz[b]].tobytes() for b in range(blk, blk + nb)); blk += nb
        assert mine == body, f0
    assert ip == len(comp) and blk == nblk


@pytest.mark.parametrize("fl,sl,opt", [(18, 1, True), (17, 0, False), (18, 0, True)])
def test_emulated_method21_pipeline_end_to_end(pkg, emu, fl, sl, opt):
    """every kernel of the method-21 encoder and decoder, as sources, in sequence: stage C -> stage P (or the oracle's stage M
    sequences for the greedy parse) -> stage R -> offsets + gather = the oracle's stream byte for byte (both placements of the
    literal model); lzma2_walk_kernel + lzma2_decode_kernel restore the input from it"""
    data = _mixed(pkg, 250_000); n = len(data)
    flags = 1 | (sl << 8) | (OPT if opt else 0)
    src = np.frombuffer(data + bytes(64), dtype=np.uint8)
    F = 1 << fl; nfr = (n + F - 1) // F; bpf = F >> 17
    if opt:
        cand = np.zeros(nfr * F * 4, dtype=np.uint32)
        emu.emu_lzma2_cand(src.ctypes.data, n, fl, flags, 2, cand.ctypes.data)
        seqs = np.zeros(nfr * bpf * H.MAXSEQ, dtype=np.uint64); nseq = np.zeros(nfr * bpf, dtype=np.uint32)
        emu.emu_lzma2_parse(src.ctypes.data, n, fl, flags, cand.ctypes.data, seqs.ctypes.data, nseq.ctypes.data)
    else:
        seqs, nseq, _, _ = H.oracle_find_sequences(data, frameLog=fl, windowLog=fl)
    prop, want = H.oracle_lzma2_compress(data, frameLog=fl, windowLog=fl, flags=flags)
    for glit in (0, 1, 2):                                              # 2 = 32 chains per warp in lock-step (lzma2_enc_range32_kernel)
        out = np.zeros(len(want) + 200_000, dtype=np.uint8)
        r = emu.emu_lzma2_range_and_assemble(src.ctypes.data, n, fl, flags, seqs.ctypes.data, nseq.ctypes.data, out.ctypes.data, out.size, glit)
        assert r == len(want) and out[:r].tobytes() == want, glit
    lz = np.frombuffer(want, dtype=np.uint8)
    for glit in (0, 1):
        back = np.zeros(n + 64, dtype=np.uint8)
        assert emu.emu_lzma2_decode(lz.ctypes.data, len(want), prop, back.ctypes.data, n, glit) == n and back[:n].tobytes() == data, glit
    # a stream of the reference's own encoder through the emulated decoder
    if H.ref_lzma_available():
        rprop, rlz = H.ref_lzma2_compress(data, level=5, dict_size=1 << 18, block_size=1 << 18)
        a = np.frombuffer(rlz, dtype=np.uint8); back = np.zeros(n + 64, dtype=np.uint8)
        assert emu.emu_lzma2_decode(a.ctypes.data, len(rlz), rprop, back.ctypes.data, n, 0) == n and back[:n].tobytes() == data


@pytest.mark.parametrize("fl,flags", [(18, 1), (17, 3), (18, 3 | ZOPT), (17, 1 | ZOPT)])
def test_emulated_zstd_encoder_end_to_end(pkg, emu, fl, flags):
    """every kernel of the Zstandard encoder, as sources, in sequence: stage M (or stage C + stage Z) -> stage E -> checksum /
    offsets / gather = the oracle's frames byte for byte (size hints, XXH64 content checksums), which the reference decoder restores"""
    data = _mixed(pkg, 300_000) + bytes(140_000); n = len(data)
    src = np.frombuffer(data + bytes(64), dtype=np.uint8)
    F = 1 << fl; nfr = (n + F - 1) // F; nblk = (n + 131071) // 131072
    seqs = np.zeros(nblk * H.MAXSEQ, dtype=np.uint64); nseq = np.zeros(nblk, dtype=np.uint32); nlit = np.zeros(nblk, dtype=np.uint32); lits = np.zeros(n + 64, dtype=np.uint8)
    if flags & ZOPT:
        cand = np.zeros(nfr * F * 4, dtype=np.uint32)
        emu.emu_lzma2_cand(src.ctypes.data, n, fl, flags, 2, cand.ctypes.data)
        emu.emu_zstd_enc_parse(src.ctypes.data, n, fl, flags, cand.ctypes.data, seqs.ctypes.data, nseq.ctypes.data, lits.ctypes.data, nlit.ctypes.data)
    else:
        emu.emu_zstd_enc_match(src.ctypes.data, n, fl, fl, 7, flags, 2, seqs.ctypes.data, nseq.ctypes.data, lits.ctypes.data, nlit.ctypes.data)
    SLOT = emu.emu_slot_bytes()
    slots = np.zeros(nblk * SLOT, dtype=np.uint8); ssz = np.zeros(nblk, dtype=np.uint32)
    emu.emu_zstd_enc_entropy(src.ctypes.data, n, fl, flags, seqs.ctypes.data, nseq.ctypes.data, lits.ctypes.data, nlit.ctypes.data, slots.ctypes.data, ssz.ctypes.data, nblk)
    want = H.oracle_compress(data, frameLog=fl, windowLog=fl, flags=flags)
    out = np.zeros(len(want) + 100_000, dtype=np.uint8)
    r = emu.emu_zstd_enc_assemble(src.ctypes.data, n, fl, flags, slots.ctypes.data, ssz.ctypes.data, nblk, out.ctypes.data, out.size)
    assert r == len(want) and out[:r].tobytes() == want
    assert H.ref_zstd_result(want, n) == H.digest(data)


def test_emulated_zstd_decoder_on_golden_and_reference_frames(pkg, emu):
    """the Zstandard decoder's kernels (frame discovery, block index, table + stream entropy kernels, layout, execute, checksum
    verify), as sources in the order dec_impl launches them: the committed golden frames written by the reference encoder
    (levels -5 .. 19, checksums, the reference's own regression archives' streams), fresh reference-encoder output, and our
    own frames of both parses"""
    import hashlib, json
    golden = os.path.join(HERE, "golden")

    def dec(comp, n):
        src = np.frombuffer(comp + bytes(64), dtype=np.uint8); dst = np.zeros(n + 64, dtype=np.uint8)
        r = emu.emu_zstd_decode(src.ctypes.data, len(comp), dst.ctypes.data, n)
        return r, dst[:max(r, 0)].tobytes()
    for idx_name in ("frames.json", "regr.json"):
        for name, meta in json.load(open(os.path.join(golden, idx_name))).items():
            if not name.endswith(".zst"):
                continue
            r, out = dec(open(os.path.join(golden, name), "rb").read(), meta["size"])
            assert r == meta["size"] and hashlib.sha256(out).hexdigest() == meta["sha256"], name
    data = _mixed(pkg, 200_000); n = len(data)
    streams = [H.oracle_compress(data), H.oracle_compress(data, flags=3 | ZOPT, frameLog=17, windowLog=17)]
    if H.ref_available():
        streams += [H.ref_compress(data, level=1), H.ref_compress(data, level=19, checksum=1), H.ref_compress(data, level=5, nbWorkers=2)]
    for k, comp in enumerate(streams):
        assert dec(comp, n) == (n, data), k
    bad = bytearray(streams[1]); bad[len(bad) // 2] ^= 0x20          # damage: an error status or a checksum mismatch, never a wrong "success"
    r, out = dec(bytes(bad), n)
    assert not (r == n and out == data)
    # a skippable frame that only LOOKS like mcmilk's size hint (0x184D2A50, 4 bytes of payload >= 9 that are not the next frame's size)
    # is user data: the stream is walked again without hints and decodes, as with the reference (which never reads hints)
    import struct
    fake = struct.pack("<III", 0x184D2A50, 4, 4242)
    assert dec(fake + streams[0] + fake + streams[1], 2 * n) == (2 * n, data + data)
    # a window descriptor far beyond what the decoder's offsets cover (2^30, 2^31) is fine when the declared content is small: no offset can
    # exceed the content (zstd_decompress.c:482-560 only bounds the window by ZSTD_WINDOWLOG_MAX); without a content size it stays unsupported
    if H.ref_available():
        f = bytearray(H.ref_compress(data, level=3, windowLog=17))
        assert f[4] & 0x20 == 0 and f[4] >> 6                       # not single-segment, content size present
        for wd in (0xA0, 0xA8):
            f[5] = wd
            assert dec(bytes(f), n) == (n, data), hex(wd)
        g = bytearray(H.ref_compress(data, level=3, windowLog=17, contentSizeFlag=0)); g[5] = 0xA8
        assert dec(bytes(g), n)[0] == -2                            # B2Z_DERR_UNSUPPORTED


def test_emulated_zstd_decoder_frames_of_several_units(pkg, emu):
    """frames longer than one execution unit (8 blocks): every unit starts from the repcode history stage D2 derived from the blocks'
    symbolic histories, and a match that reaches behind its unit waits for the unit that wrote the bytes.  Reference-written frames
    with a sliding window (repcodes and matches cross every unit boundary), a frame of this encoder's long mode (far matches into
    other regions), blocks of zeros (RLE), noise (raw blocks) and repcode-only stretches in between"""
    def dec(comp, n):
        src = np.frombuffer(comp + bytes(64), dtype=np.uint8); dst = np.zeros(n + 64, dtype=np.uint8)
        r = emu.emu_zstd_decode(src.ctypes.data, len(comp), dst.ctypes.data, n)
        return r, dst[:max(r, 0)].tobytes()
    data = (H.far_copies(pkg, (3 << 20) + 777, every=1 << 19, span=(30_000, 90_000), seed=2) + bytes(300_000) + pkg.corpus.entropy_class(1, 200_000).tobytes()
            + b"abcdefghij" * 40_000 + pkg.corpus.g2(400_000).tobytes())
    n = len(data)
    streams = [H.oracle_compress(data, frameLog=23, windowLog=23, regionLog=18, ldmLog=14), H.oracle_compress(data, frameLog=22, windowLog=22)]
    if H.ref_available():
        streams += [H.ref_compress(data, level=3), H.ref_compress(data, level=1, checksum=1), H.ref_compress(data, level=12),
                    H.ref_compress(data, level=3, windowLog=23, enableLongDistanceMatching=1)]
    for k, comp in enumerate(streams):
        r, out = dec(comp, n)
        assert r == n and out == data, k


def test_emulated_zstd_decoder_scratch_follows_compressed_blocks(pkg, emu):
    """raw and RLE blocks own no literal / sequence scratch (DecBlock::slot numbers the compressed blocks only): a reference frame of
    128 RLE blocks of zeros, 16 raw blocks of noise and a little text decodes with scratch for the text's blocks alone -- through the
    execution units and through stage J"""
    if not H.ref_available():
        pytest.skip("oracle/_ref not built")
    data = bytes(16 << 20) + pkg.corpus.entropy_class(1, 2 << 20).tobytes() + pkg.corpus.g2(300_000).tobytes() + bytes(1 << 20); n = len(data)
    comp = H.ref_compress(data, level=3)
    src = np.frombuffer(comp + bytes(64), dtype=np.uint8)
    for mode in (0, 2):
        dst = np.full(n + 64, 0xEE, dtype=np.uint8); nj = ctypes.c_uint32(0)
        r = emu.emu_zstd_decode_jump(src.ctypes.data, len(comp), dst.ctypes.data, n, mode, ctypes.byref(nj))
        assert r == n and dst[:n].tobytes() == data, mode


def test_emulated_zstd_decoder_stage_j_pointer_jumping(pkg, emu):
    """stage J (zstd_dec_jump_build / _round kernels): literal bytes + one pointer per output byte, pointer doubling, byte gather.
    Forced on every frame (mode 2) it must give what the execution units give -- golden frames of the reference encoder, frames with
    raw / RLE blocks, long runs (offset 1: the chain inside a match is cut by the periodic source), repcodes across blocks, several
    frames in one stream, damaged streams; in automatic mode (1) a reference-written sliding-window frame of >= 8 units is taken by
    stage J and frames of this encoder (independent regions, or too short) are not"""
    import hashlib, json
    def dec(comp, n, mode):
        src = np.frombuffer(comp + bytes(64), dtype=np.uint8); dst = np.full(n + 64, 0xEE, dtype=np.uint8); nj = ctypes.c_uint32(0)
        r = emu.emu_zstd_decode_jump(src.ctypes.data, len(comp), dst.ctypes.data, n, mode, ctypes.byref(nj))
        return r, dst[:max(r, 0)].tobytes(), nj.value
    golden = os.path.join(HERE, "golden")
    emu.emu_set_jump_seglog.argtypes = [ctypes.c_uint32]; emu.emu_set_jump_seglog.restype = None
    emu.emu_set_jump_seglog(30)
    for idx_name in ("frames.json", "regr.json"):
        for name, meta in json.load(open(os.path.join(golden, idx_name))).items():
            if not name.endswith(".zst"):
                continue
            r, out, nj = dec(open(os.path.join(golden, name), "rb").read(), meta["size"], 2)
            assert r == meta["size"] and hashlib.sha256(out).hexdigest() == meta["sha256"] and (nj > 0 or r == 0), name
    data = _mixed(pkg, 300_000) + bytes(400_000) + b"abcdefghij" * 30_000 + pkg.corpus.g2(200_000).tobytes(); n = len(data)
    streams = [H.oracle_compress(data), H.oracle_compress(data, frameLog=22, windowLog=22), H.oracle_compress(data, flags=3 | ZOPT, frameLog=17, windowLog=17)]
    if H.ref_available():
        streams += [H.ref_compress(data, level=1), H.ref_compress(data, level=19, checksum=1), H.ref_compress(data, level=5, nbWorkers=2)]
    for k, comp in enumerate(streams):
        r, out, nj = dec(comp, n, 2)
        assert (r, out) == (n, data) and nj > 0, k
        assert dec(comp, n, 0) == (n, data, 0), k
    bad = bytearray(streams[1]); bad[len(bad) // 2] ^= 0x20
    r, out, nj = dec(bytes(bad), n, 2)
    assert not (r == n and out == data)
    # segments: the output resolved in pieces of 64 KiB / 128 KiB, in order (what lets a frame of any size through 31-bit pointers): blocks
    # straddle the cuts, sources lie segments back
    for seglog in (16, 17):
        emu.emu_set_jump_seglog(seglog)
        for k, comp in enumerate(streams):
            r, out, nj = dec(comp, n, 2)
            assert (r, out) == (n, data) and nj > 0, (seglog, k)
    emu.emu_set_jump_seglog(30)
    # automatic mode: 5 MiB, one frame
    big = pkg.corpus.g2(5 << 20).tobytes() + b"q" * 70_000; nb = len(big)
    ours = H.oracle_compress(big, frameLog=23, windowLog=23, regionLog=19, ldmLog=14)
    r, out, nj = dec(ours, nb, 1)
    assert (r, out) == (nb, big) and nj == 0                     # regions are independent: the units run side by side
    if H.ref_available():
        ref = H.ref_compress(big, level=3)
        r, out, nj = dec(ref, nb, 1)
        assert (r, out) == (nb, big) and nj == 1                 # one sliding-window frame: stage J
        r, out, nj = dec(ref + H.oracle_compress(data) + ref, 2 * nb + n, 1)
        assert (r, out) == (2 * nb + n, big + data + big) and nj == 2
        # half the frame is RLE blocks: the text half is still a chain of six units -- three consecutive chained units are enough
        half = bytes(3 << 20) + pkg.corpus.g2(3 << 20).tobytes()
        for lv in (1, 9):
            r, out, nj = dec(H.ref_compress(half, level=lv), len(half), 1)
            assert (r, out) == (len(half), half) and nj == 1, lv


def test_emulated_stage_z_sequence_array_full(pkg, emu):
    """a block whose parse wants more sequences than its array holds (32 768; random 3-byte tokens give one length-3 match every
    three bytes): from there on the matches' bytes stay literals -- the same rule in the oracle and the kernel, and the frame decodes"""
    import random
    rng = random.Random(1)
    toks = [bytes(rng.randrange(256) for _ in range(3)) for _ in range(64)]
    data = b"".join(rng.choice(toks) for _ in range(90_000))[:2 * 131072 + 5000]; n = len(data); fl = 18
    src = np.frombuffer(data + bytes(64), dtype=np.uint8)
    zs, zn, zl, znl = H.oracle_find_sequences(data, frameLog=fl, windowLog=fl, flags=1 | ZOPT)
    assert int(zn[0]) == H.MAXSEQ                                   # the case this test is about
    nfr = (n + (1 << fl) - 1) >> fl
    cand = np.zeros(nfr * (1 << fl) * 4, dtype=np.uint32)
    emu.emu_lzma2_cand(src.ctypes.data, n, fl, 1, 1, cand.ctypes.data)
    seqZ = np.zeros_like(zs); nsZ = np.zeros_like(zn); nlZ = np.zeros_like(znl); litZ = np.zeros(n + 64, dtype=np.uint8)
    emu.emu_zstd_enc_parse(src.ctypes.data, n, fl, 1 | ZOPT, cand.ctypes.data, seqZ.ctypes.data, nsZ.ctypes.data, litZ.ctypes.data, nlZ.ctypes.data)
    assert np.array_equal(nsZ, zn) and np.array_equal(nlZ, znl)
    for b in range(len(zn)):
        assert np.array_equal(seqZ[b * H.MAXSEQ:b * H.MAXSEQ + zn[b]], zs[b * H.MAXSEQ:b * H.MAXSEQ + zn[b]]), b
        assert np.array_equal(litZ[b * 131072:b * 131072 + znl[b]], zl[b * 131072:b * 131072 + znl[b]]), b
    comp = H.oracle_compress(data, frameLog=fl, windowLog=fl, flags=1 | ZOPT)
    assert H.oracle_decompress(comp, n) == data
    assert H.ref_zstd_result(comp, n) == H.digest(data)
    # 32 768 sequences take the 3-byte form of the sequence count (>= 0x7F00): stage E writes it, the decoder kernels read it
    nblk = len(zn); SLOT = emu.emu_slot_bytes()
    lits = np.zeros(n + 64, dtype=np.uint8); lits[:n] = zl
    slots = np.zeros(nblk * SLOT, dtype=np.uint8); ssz = np.zeros(nblk, dtype=np.uint32)
    emu.emu_zstd_enc_entropy(src.ctypes.data, n, fl, 1 | ZOPT, zs.ctypes.data, zn.ctypes.data, lits.ctypes.data, znl.ctypes.data, slots.ctypes.data, ssz.ctypes.data, nblk)
    out = np.zeros(len(comp) + 100_000, dtype=np.uint8)
    r = emu.emu_zstd_enc_assemble(src.ctypes.data, n, fl, 1 | ZOPT, slots.ctypes.data, ssz.ctypes.data, nblk, out.ctypes.data, out.size)
    assert r == len(comp) and out[:r].tobytes() == comp
    c = np.frombuffer(comp + bytes(64), dtype=np.uint8); back = np.zeros(n + 64, dtype=np.uint8)
    assert emu.emu_zstd_decode(c.ctypes.data, len(comp), back.ctypes.data, n) == n and back[:n].tobytes() == data


def test_emulated_capped_candidate_is_clipped_at_the_boundary(pkg, emu):
    data = H.capped_match_near_boundary(pkg); n = len(data); fl = 18
    src = np.frombuffer(data + bytes(64), dtype=np.uint8)
    F = 1 << fl; nfr = (n + F - 1) // F; bpf = F >> 17
    cand = np.zeros(nfr * F * 4, dtype=np.uint32)
    emu.emu_lzma2_cand(src.ctypes.data, n, fl, 1, 1, cand.ctypes.data)
    assert int((cand & 0xFF).max()) == 255                          # there are capped words
    # stage Z (block boundary)
    zs, zn, zl, znl = H.oracle_find_sequences(data, frameLog=fl, windowLog=fl, flags=1 | ZOPT)
    seqZ = np.zeros_like(zs); nsZ = np.zeros_like(zn); nlZ = np.zeros_like(znl); litZ = np.zeros(n + 64, dtype=np.uint8)
    emu.emu_zstd_enc_parse(src.ctypes.data, n, fl, 1 | ZOPT, cand.ctypes.data, seqZ.ctypes.data, nsZ.ctypes.data, litZ.ctypes.data, nlZ.ctypes.data)
    assert np.array_equal(nsZ, zn) and np.array_equal(nlZ, znl)
    for b in range(len(zn)):
        assert np.array_equal(seqZ[b * H.MAXSEQ:b * H.MAXSEQ + zn[b]], zs[b * H.MAXSEQ:b * H.MAXSEQ + zn[b]]), b
    ml0 = [H.seq_fields(s)[2] for s in zs[:zn[0]]]; ml1 = [H.seq_fields(s)[2] for s in zs[H.MAXSEQ:H.MAXSEQ + zn[1]]]
    assert any(90 <= m <= 100 for m in ml0) and max(ml0) <= 100       # the capped candidate clipped at the block end ...
    assert 300 in ml1 and max(ml1) > 3000                             # ... and capped candidates extended past 255 where there is room
    # stage P (slice boundary: two slices of 128 KiB per 256 KiB frame)
    flags = 1 | (1 << 8) | OPT
    candO, seqO, nsO = _oracle_taps(data, fl, flags)
    seqE = np.zeros_like(seqO); nsE = np.zeros_like(nsO)
    emu.emu_lzma2_parse(src.ctypes.data, n, fl, flags, cand.ctypes.data, seqE.ctypes.data, nsE.ctypes.data)
    assert np.array_equal(nsE, nsO)
    for b in range(len(nsO)):
        assert np.array_equal(seqE[b * H.MAXSEQ:b * H.MAXSEQ + nsO[b]], seqO[b * H.MAXSEQ:b * H.MAXSEQ + nsO[b]]), b
    prop, lz = H.oracle_lzma2_compress(data, frameLog=fl, windowLog=fl, flags=flags)
    assert H.oracle_lzma2_decompress(lz, n, prop)[0] == data
    assert H.ref_lzma2_result(lz, n, prop)[0] == H.digest(data)
