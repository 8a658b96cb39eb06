"""CPU: seeded structured-random inputs (noise, runs, tiny alphabets, periodic data with mutations, word text, G2 text; sizes around
the 32-lane step, the 256-node window and the 128 KiB block) through the emulated kernel sources of stage C / stage P / stage Z
against the oracle, and the resulting streams through the reference's decoders.  (Longer runs of the same generators with other seeds,
also under AddressSanitizer -- 3 500 inputs -- found one difference, the boundary bug fixed in the long-match path; this is the bounded version.)  See tests/cuemu/cuemu.h for what the emulation is."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import helpers as H

HERE = os.path.dirname(os.path.abspath(__file__))
SIZES = [1, 2, 3, 5, 31, 32, 33, 255, 256, 257, 1000, 4097, 20000, 70000, 131072, 131073, 140000]


def _planted(rng, pkg):
    """noise / text with planted copies of many lengths, some ending or starting around the 128 KiB block and slice boundaries and
    around the 255-byte cap of stage C's stored lengths (this shape found the boundary bug of the long-match path)"""
    n = rng.choice([140000, 262144 + 7, 131072 + 300])
    a = bytearray(pkg.corpus.entropy_class(1, n).tobytes() if rng.random() < 0.6 else pkg.corpus.g2(n, seed=rng.randrange(99)).tobytes())
    for _ in range(rng.randrange(3, 40)):
        L = rng.choice([20, 33, 100, 223, 224, 255, 256, 273, 274, 300, 1000, 5000]); srcp = rng.randrange(0, n - L)
        if rng.random() < 0.5:
            dstp = rng.choice([131072, 262144]) - rng.choice([0, 1, 31, 32, 33, 99, 100, 223, 224, 225, 254, 255, 256, 272, 273, 274, 300]) + rng.choice([0, 0, 0, 500])
        else:
            dstp = rng.randrange(0, n - L)
        if 0 <= dstp and dstp + L <= n and dstp > srcp:
            a[dstp:dstp + L] = a[srcp:srcp + L]
    return bytes(a)


def _gen(rng, pkg, planted=False):
    if planted:
        return _planted(rng, pkg)
    kind = rng.randrange(6); n = rng.choice(SIZES)
    if kind == 0:
        return bytes(rng.randrange(256) for _ in range(min(n, 30000)))
    if kind == 1:
        return bytes([rng.randrange(3)]) * n
    if kind == 2:
        alpha = bytes(rng.randrange(256) for _ in range(rng.choice([2, 3, 4, 16])))
        return bytes(rng.choice(alpha) for _ in range(min(n, 60000)))
    if kind == 3:
        unit = bytes(rng.randrange(256) for _ in range(rng.choice([1, 2, 3, 7, 31, 33, 100, 300, 5000])))
        out = bytearray((unit * (n // len(unit) + 1))[:n])
        for _ in range(n // 200 + 1):
            out[rng.randrange(n)] = rng.randrange(256)
        return bytes(out)
    if kind == 4:
        return pkg.corpus.g2(n, seed=rng.randrange(1000)).tobytes()
    words = [bytes(rng.randrange(97, 123) for _ in range(rng.randrange(1, 9))) for _ in range(rng.choice([5, 50, 500]))]
    out = bytearray()
    while len(out) < n:
        out += rng.choice(words) + b" "
    return bytes(out[:n])


@pytest.mark.parametrize("seed", [11, 12, 13, 41])
def test_fuzz_emulated_kernels_equal_the_oracle(pkg, seed):
    E = H.cuemu_library()
    vp, u32, u64 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64
    E.emu_zstd_enc_parse.restype = u64; E.emu_zstd_enc_parse.argtypes = [vp, u64, u32, u32, vp, vp, vp, vp, vp]
    E.emu_lzma2_cand.restype = u64; E.emu_lzma2_cand.argtypes = [vp, u64, u32, u32, u32, vp]
    E.emu_lzma2_parse.restype = u64; E.emu_lzma2_parse.argtypes = [vp, u64, u32, u32, vp, vp, vp]
    O = H.oracle()
    O.b2zo_lzma2_candidates.argtypes = [vp, u32, u32, vp]
    O.b2zo_lzma2_parse_frame.argtypes = [vp, u32, ctypes.POINTER(H.EncParams), vp, vp, vp]
    rng = random.Random(seed)
    for it in range(14 if seed < 40 else 2):                       # seeds >= 40: the (larger) planted-copy inputs
        data = _gen(rng, pkg, planted=seed >= 40); n = len(data)
        fl = rng.choice([17, 17, 18]); sl = rng.choice([0, 1]) if fl == 18 else 0
        F = 1 << fl; nfr = (n + F - 1) // F; bpf = F >> 17
        src = np.frombuffer(data + bytes(64), dtype=np.uint8)
        candO = np.zeros(nfr * F * 4, dtype=np.uint32)
        for f in range(nfr):
            O.b2zo_lzma2_candidates(src.ctypes.data + f * F, min(F, n - f * F), fl, candO.ctypes.data + f * F * 16)
        candE = np.zeros_like(candO)
        E.emu_lzma2_cand(src.ctypes.data, n, fl, 1, rng.choice([1, 2, 3]), candE.ctypes.data)
        assert np.array_equal(candE[:n * 4], candO[:n * 4]), ("stage C", seed, it, n, fl)
        flags = 1 | (sl << 8) | 0x10
        p = H.enc_params(frameLog=fl, windowLog=fl, flags=flags)
        seqO = np.zeros(nfr * bpf * H.MAXSEQ, dtype=np.uint64); nsO = np.zeros(nfr * bpf, dtype=np.uint32)
        for f in range(nfr):
            O.b2zo_lzma2_parse_frame(src.ctypes.data + f * F, min(F, n - f * F), ctypes.byref(p), candO.ctypes.data + f * F * 16,
                                     seqO.ctypes.data + f * bpf * H.MAXSEQ * 8, nsO.ctypes.data + f * bpf * 4)
        seqE = np.zeros_like(seqO); nsE = np.zeros_like(nsO)
        E.emu_lzma2_parse(src.ctypes.data, n, fl, flags, candO.ctypes.data, seqE.ctypes.data, nsE.ctypes.data)
        nb = (n + 131071) // 131072
        assert np.array_equal(nsE[:nb], nsO[:nb]), ("stage P counts", seed, it, n, fl, sl)
        for b in range(nb):
            assert np.array_equal(seqE[b * H.MAXSEQ:b * H.MAXSEQ + nsO[b]], seqO[b * H.MAXSEQ:b * H.MAXSEQ + nsO[b]]), ("stage P", seed, it, n, b)
        zs, zn, zl, znl = H.oracle_find_sequences(data, frameLog=fl, windowLog=fl, flags=1 | 0x20)
        seqZ = np.zeros_like(zs); nsZ = np.full_like(zn, 0xFFFFFFFF); nlZ = np.full_like(znl, 0xFFFFFFFF); litZ = np.zeros(n + 64, dtype=np.uint8)
        E.emu_zstd_enc_parse(src.ctypes.data, n, fl, 1 | 0x20, candO.ctypes.data, seqZ.ctypes.data, nsZ.ctypes.data, litZ.ctypes.data, nlZ.ctypes.data)
        assert np.array_equal(nsZ, zn) and np.array_equal(nlZ, znl), ("stage Z counts", seed, it, n, fl)
        for b in range(len(zn)):
            assert np.array_equal(seqZ[b * H.MAXSEQ:b * H.MAXSEQ + zn[b]], zs[b * H.MAXSEQ:b * H.MAXSEQ + zn[b]]), ("stage Z sequences", seed, it, n, b)
            assert np.array_equal(litZ[b * 131072:b * 131072 + znl[b]], zl[b * 131072:b * 131072 + znl[b]]), ("stage Z literals", seed, it, n, b)
        comp = H.oracle_compress(data, frameLog=fl, windowLog=fl, flags=1 | 0x20)
        assert H.ref_zstd_result(comp, n) == H.digest(data)
        prop, lz = H.oracle_lzma2_compress(data, frameLog=fl, windowLog=fl, flags=flags)
        assert H.ref_lzma2_result(lz, n, prop)[0] == H.digest(data)


@pytest.mark.parametrize("seed,planted", [(51, False), (52, True)])
def test_fuzz_emulated_pipelines_and_damaged_streams(pkg, seed, planted):
    """the hardware-verified kernels through the same generators: stage M -> stage E -> assembly == the oracle's frames, stage R ->
    assembly == the oracle's chunk stream, the decoder kernels restore both -- and on DAMAGED streams (bit flips, overwritten
    bytes, deletions, truncation) they end with an error status or some output, never with a wild access (longer runs of this
    loop under AddressSanitizer: 2 100 inputs, 13 000 decodes, no report)"""
    E = H.cuemu_library()
    vp, u32, u64, i64 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int64
    E.emu_zstd_enc_match.restype = u64; E.emu_zstd_enc_match.argtypes = [vp, u64, u32, u32, u32, u32, u32, vp, vp, vp, vp]
    E.emu_zstd_enc_entropy.restype = u64; E.emu_zstd_enc_entropy.argtypes = [vp, u64, u32, u32, vp, vp, vp, vp, vp, vp, u32]
    E.emu_slot_bytes.restype = u32
    E.emu_zstd_enc_assemble.restype = i64; E.emu_zstd_enc_assemble.argtypes = [vp, u64, u32, u32, vp, vp, u32, vp, u64]
    E.emu_zstd_decode.restype = i64; E.emu_zstd_decode.argtypes = [vp, u64, vp, u64]
    E.emu_lzma2_range_and_assemble.restype = i64; E.emu_lzma2_range_and_assemble.argtypes = [vp, u64, u32, u32, vp, vp, vp, u64, ctypes.c_int]
    E.emu_lzma2_decode.restype = i64; E.emu_lzma2_decode.argtypes = [vp, u64, u32, vp, u64, ctypes.c_int]
    E.emu_zstd_decode_jump.restype = i64; E.emu_zstd_decode_jump.argtypes = [vp, u64, vp, u64, u32, vp]
    E.emu_set_jump_seglog.restype = None; E.emu_set_jump_seglog.argtypes = [u32]
    SLOT = E.emu_slot_bytes(); rng = random.Random(seed)
    for it in range(5 if planted else 12):
        data = _gen(rng, pkg, planted); n = len(data)
        fl = rng.choice([17, 17, 18]); sl = rng.choice([0, 1]) if fl == 18 else 0
        src = np.frombuffer(data + bytes(64), dtype=np.uint8)
        nblk = (n + 131071) // 131072; F = 1 << fl; nfr = (n + F - 1) // F; bpf = F >> 17
        flagsz = rng.choice([1, 3])
        seqs = np.zeros(nblk * H.MAXSEQ, dtype=np.uint64); nseq = np.zeros(nblk, dtype=np.uint32); nlit = np.zeros(nblk, dtype=np.uint32); lits = np.zeros(n + 64, dtype=np.uint8)
        E.emu_zstd_enc_match(src.ctypes.data, n, fl, fl, 7, flagsz, rng.choice([1, 2]), seqs.ctypes.data, nseq.ctypes.data, lits.ctypes.data, nlit.ctypes.data)
        slots = np.zeros(nblk * SLOT, dtype=np.uint8); ssz = np.zeros(nblk, dtype=np.uint32)
        E.emu_zstd_enc_entropy(src.ctypes.data, n, fl, flagsz, seqs.ctypes.data, nseq.ctypes.data, lits.ctypes.data, nlit.ctypes.data, slots.ctypes.data, ssz.ctypes.data, nblk)
        want = H.oracle_compress(data, frameLog=fl, windowLog=fl, flags=flagsz)
        out = np.zeros(len(want) + 100_000, dtype=np.uint8)
        r = E.emu_zstd_enc_assemble(src.ctypes.data, n, fl, flagsz, slots.ctypes.data, ssz.ctypes.data, nblk, out.ctypes.data, out.size)
        assert r == len(want) and out[:r].tobytes() == want, ("zstd M -> E -> assemble", seed, it, n, fl, flagsz)
        flagsl = 1 | (sl << 8)
        so, no, _, _ = H.oracle_find_sequences(data, frameLog=fl, windowLog=fl, flags=flagsl)
        prop, wantl = H.oracle_lzma2_compress(data, frameLog=fl, windowLog=fl, flags=flagsl)
        seqf = np.zeros(nfr * bpf * H.MAXSEQ, dtype=np.uint64); nsf = np.zeros(nfr * bpf, dtype=np.uint32); b = 0
        for f in range(nfr):                                        # the oracle's tap numbers blocks densely; stage R per frame
            for k in range((min(F, n - f * F) + 131071) // 131072):
                seqf[(f * bpf + k) * H.MAXSEQ:(f * bpf + k + 1) * H.MAXSEQ] = so[b * H.MAXSEQ:(b + 1) * H.MAXSEQ]; nsf[f * bpf + k] = no[b]; b += 1
        outl = np.zeros(len(wantl) + 200_000, dtype=np.uint8)
        r = E.emu_lzma2_range_and_assemble(src.ctypes.data, n, fl, flagsl, seqf.ctypes.data, nsf.ctypes.data, outl.ctypes.data, outl.size, rng.choice([0, 1, 2, 2]))
        assert r == len(wantl) and outl[:r].tobytes() == wantl, ("lzma2 R -> assemble", seed, it, n, fl, sl)
        for comp, kind in ((want, "z"), (wantl, "l")):
            for mut in range(3):
                c = bytearray(comp)
                if mut:
                    for _ in range(rng.choice([1, 1, 3])):
                        k = rng.randrange(4)
                        if k == 0 and c: c[rng.randrange(len(c))] ^= 1 << rng.randrange(8)
                        elif k == 1 and c: c[rng.randrange(len(c))] = rng.randrange(256)
                        elif k == 2 and len(c) > 4: del c[rng.randrange(len(c)):rng.randrange(len(c)) + rng.randrange(1, 9)]
                        else: c = c[:rng.randrange(len(c) + 1)]
                cb = np.frombuffer(bytes(c) + bytes(64), dtype=np.uint8); back = np.zeros(n + 64, dtype=np.uint8)
                if kind == "z":
                    if rng.random() < 0.5:                          # stage J forced on every frame, the output resolved in small segments
                        E.emu_set_jump_seglog(rng.choice([16, 17, 30]))
                        r = E.emu_zstd_decode_jump(cb.ctypes.data, len(c), back.ctypes.data, n, 2, None)
                    else:
                        r = E.emu_zstd_decode(cb.ctypes.data, len(c), back.ctypes.data, n)
                else:
                    r = E.emu_lzma2_decode(cb.ctypes.data, len(c), prop, back.ctypes.data, n, rng.choice([0, 1, 2, 2])) if len(c) else -1
                if not mut:
                    assert r == n and back[:n].tobytes() == data, ("decode", kind, seed, it, n)
                else:
                    assert r <= n                                   # an error status (< 0) or at most the declared output


def test_emulated_decoders_give_the_oracle_decoders_verdict_on_damaged_streams(pkg):
    """same accept / reject decision and the same bytes as the oracle decoders (which are pinned to the reference decoders' behaviour
    on corrupt input) for bit flips, overwritten bytes and truncation (6 000 mutants in a longer run: no difference)"""
    E = H.cuemu_library()
    vp, u32, u64, i64 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int64
    E.emu_lzma2_decode.restype = i64; E.emu_lzma2_decode.argtypes = [vp, u64, u32, vp, u64, ctypes.c_int]
    E.emu_zstd_decode.restype = i64; E.emu_zstd_decode.argtypes = [vp, u64, vp, u64]
    E.emu_zstd_decode_jump.restype = i64; E.emu_zstd_decode_jump.argtypes = [vp, u64, vp, u64, u32, vp]
    E.emu_set_jump_seglog.restype = None; E.emu_set_jump_seglog.argtypes = [u32]
    data = pkg.corpus.g2(120_000).tobytes() + bytes(3000) + pkg.corpus.entropy_class(1, 30_000).tobytes(); n = len(data)
    prop, lz = H.oracle_lzma2_compress(data, frameLog=17, windowLog=17, flags=1)
    zs = H.oracle_compress(data, frameLog=17, windowLog=17, flags=3)
    rng = random.Random(3)
    for it in range(250):
        for kind, comp in (("l", lz), ("z", zs)):
            c = bytearray(comp); k = rng.randrange(3)
            if k == 0:
                c[rng.randrange(len(c))] ^= 1 << rng.randrange(8)
            elif k == 1:
                c[rng.randrange(len(c))] = rng.randrange(256)
            else:
                c = c[:rng.randrange(1, len(c))]
            cb = np.frombuffer(bytes(c) + bytes(64), dtype=np.uint8); back = np.zeros(n + 64, dtype=np.uint8)
            try:
                want = H.oracle_lzma2_decompress(bytes(c), n, prop)[0] if kind == "l" else H.oracle_decompress(bytes(c), n)
            except ValueError:
                want = None
            if kind == "z" and it % 3 == 2:                          # every third mutant through stage J (forced), 64 KiB segments
                E.emu_set_jump_seglog(16)
                r = E.emu_zstd_decode_jump(cb.ctypes.data, len(c), back.ctypes.data, n, 2, None)
                E.emu_set_jump_seglog(30)
            else:
                r = (E.emu_lzma2_decode(cb.ctypes.data, len(c), prop, back.ctypes.data, n, it & 1) if kind == "l"
                     else E.emu_zstd_decode(cb.ctypes.data, len(c), back.ctypes.data, n))
            assert (r >= 0) == (want is not None), (kind, it, k, r)
            if want is not None:
                assert back[:r].tobytes() == want, (kind, it, k)
