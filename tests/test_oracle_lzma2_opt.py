"""CPU: oracle/lzma2_opt_oracle.c -- the price-based parse of the method-21 encoder (flag bit 4; stage C candidates + stage P
dynamic programme) writes valid LZMA2 (three independent decoders restore the input), its stage taps have the stated
properties, and the ratio moves towards the reference's optimal parsers."""
import ctypes
import lzma

import numpy as np
import pytest

import helpers as H

OPT = 0x10


def _dict_size(prop):
    return (2 | (prop & 1)) << (prop // 2 + 11)


def _candidates(data, frame_log=20):
    O = H.oracle()
    O.b2zo_lzma2_candidates.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p]
    src = np.frombuffer(data, dtype=np.uint8)
    cand = np.zeros(len(data) * 4, dtype=np.uint32)
    O.b2zo_lzma2_candidates(src.ctypes.data, len(data), frame_log, cand.ctypes.data)
    return cand.reshape(-1, 4)


def test_roundtrip_three_decoders(pkg):
    for name, data in H.sample_inputs(pkg, big=True).items():
        prop, comp = H.oracle_lzma2_compress(data, flags=1 | (2 << 8) | OPT)
        assert prop == 16 and comp[-1] == 0
        assert H.oracle_lzma2_decompress(comp, len(data), prop) == (data, len(comp)), name
        assert lzma.LZMADecompressor(format=lzma.FORMAT_RAW, filters=[{"id": lzma.FILTER_LZMA2, "dict_size": _dict_size(prop)}]).decompress(comp) == data, name
        assert H.ref_lzma2_result(comp, len(data), prop) == (H.digest(data), len(comp)), name


def test_candidates_are_nearest_previous_occurrences(pkg):
    """stage C is a pure function of the bytes: entry t of position p is the nearest q < p whose k-byte key maps to the same
    table entry (checked against a brute-force statement on a small input), with the common-prefix length (capped at 255)."""
    data = pkg.corpus.g2(40_000).tobytes() + bytes(700) + pkg.corpus.entropy_class(3, 20_000).tobytes()
    n = len(data); b = np.frombuffer(data, dtype=np.uint8)
    cand = _candidates(data, 20)
    pad = np.concatenate([b, np.zeros(8, dtype=np.uint8)])
    v = np.zeros(n, dtype=np.uint64)
    for k in range(8):
        v |= pad[k:k + n].astype(np.uint64) << np.uint64(8 * k)      # bytes past the frame end read as zero, as in the oracle
    PRIME8 = np.uint64(0xCF1BBCDCB7A56463)
    logs = {0: 16, 1: 18, 2: 19, 3: 20}; kbs = {0: 3, 1: 4, 2: 6, 3: 8}
    for t in range(4):
        kb, lg = kbs[t], logs[t]
        with np.errstate(over="ignore"):
            idx = ((v << np.uint64(64 - 8 * kb)) * PRIME8) >> np.uint64(64 - lg)
        last = {}
        for p in range(n):
            want = 0
            if p + kb <= n:
                q = last.get(int(idx[p]))
                last[int(idx[p])] = p
                if q is not None:
                    m = min(n - p, 273); l = 0
                    while l < m and data[q + l] == data[p + l]:
                        l += 1
                    if l >= 2:
                        want = ((p - q - 1) << 8) | min(l, 255)
            assert cand[p, t] == want, (p, t)


def test_parse_taps_cover_the_frame_and_reference_valid_history(pkg):
    """stage P's sequences: per block, literal runs + match lengths never run past the frame; every match copies equal bytes."""
    data = pkg.corpus.g2((1 << 20) + 77_777).tobytes()
    O = H.oracle(); p = H.enc_params(flags=1 | (2 << 8) | OPT)
    O.b2zo_lzma2_parse_frame.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.POINTER(H.EncParams), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    for f0 in (0, 1 << 20):
        frame = data[f0:f0 + (1 << 20)]; n = len(frame)
        src = np.frombuffer(frame, dtype=np.uint8)
        nblk = (n + 131071) // 131072
        seqs = np.zeros(nblk * H.MAXSEQ, dtype=np.uint64); nseq = np.zeros(nblk, dtype=np.uint32)
        O.b2zo_lzma2_parse_frame(src.ctypes.data, n, ctypes.byref(p), None, seqs.ctypes.data, nseq.ctypes.data)
        pos = 0; nm = 0
        for b in range(nblk):
            pos = max(pos, b << 17)
            for i in range(int(nseq[b])):
                s = int(seqs[b * H.MAXSEQ + i])
                ob_, ll, ml = H.seq_fields(s); off = ob_ - 3
                assert off >= 1 and 2 <= ml <= 273
                pos += ll
                assert pos - off >= 0 and pos + ml <= n
                assert all(frame[pos + k] == frame[pos + k - off] for k in range(ml))      # overlapping copies included
                pos += ml; nm += 1
        assert pos <= n and nm > n // 25


def test_ratio_moves_towards_the_reference_optimal_parsers(pkg):
    data = pkg.corpus.g2(4 << 20).tobytes()
    greedy = len(H.oracle_lzma2_compress(data)[1])
    opt = len(H.oracle_lzma2_compress(data, flags=1 | (2 << 8) | OPT)[1])
    opt1 = len(H.oracle_lzma2_compress(data, flags=1 | (0 << 8) | OPT)[1])
    opt22 = len(H.oracle_lzma2_compress(data, flags=1 | (2 << 8) | OPT, frameLog=22, windowLog=22)[1])
    assert opt < 0.955 * greedy                     # measured: 2.54 against 2.40 on G2 text
    assert opt22 < opt1 < opt
    ref_1m_blocks = H.ref_size(H.ref_lzma2_compress, data, level=5, dict_size=1 << 20, block_size=1 << 20)    # the reference's optimal parse on the same independent 1 MiB blocks
    assert opt1 < 1.03 * ref_1m_blocks
    fl2 = H.ref_size(H.ref_fl2_compress, data, 5)
    assert opt22 < 1.06 * fl2


def test_slices_and_large_frames(pkg):
    data = pkg.corpus.entropy_class(3, 3 << 20).tobytes() + bytes(2 << 20) + pkg.corpus.g2(1 << 20).tobytes() + pkg.corpus.entropy_class(1, 300_000).tobytes()
    for fl, sl in ((20, 0), (20, 3), (22, 3), (23, 1)):
        prop, comp = H.oracle_lzma2_compress(data, frameLog=fl, windowLog=fl, flags=1 | (sl << 8) | OPT)
        assert prop == (fl - 12) * 2
        assert H.oracle_lzma2_decompress(comp, len(data), prop) == (data, len(comp))
        assert H.ref_lzma2_result(comp, len(data), prop) == (H.digest(data), len(comp))


def test_simulated_model_equals_the_coders_model(pkg):
    """Stage P prices from a model it maintains itself (lzm_commit_* of csrc/b2z_lzma_model.h, the header the kernel shares); stage
    R's statement (lzma2_enc_oracle.c: enc_literal / enc_match inside the range coder) is written independently.  After the same
    packets both must hold the same probabilities, state and rep history -- the claim "the parse prices from the coder's model"."""
    O = H.oracle()
    vp, u32 = ctypes.c_void_p, ctypes.c_uint32
    O.b2zo_lzma2_final_model.restype = ctypes.c_int64
    O.b2zo_lzma2_final_model.argtypes = [vp, u32, ctypes.POINTER(H.EncParams), vp, vp, vp, vp]
    O.b2zo_lzma2_parse_final_model.argtypes = [vp, u32, ctypes.POINTER(H.EncParams), vp, vp, vp, vp]
    NP = 1848 + (0x300 << 2)
    for data, fl, sl in ((pkg.corpus.g2(300_000).tobytes(), 20, 0), (pkg.corpus.g2(600_000).tobytes() + b"abcd" * 9000, 20, 1),
                         (pkg.corpus.entropy_class(3, 200_000).tobytes(), 18, 0)):
        n = len(data); src = np.frombuffer(data, dtype=np.uint8)
        p = H.enc_params(frameLog=fl, windowLog=fl, flags=1 | (sl << 8) | OPT)
        nblk = (n + 131071) // 131072
        seqs = np.zeros(nblk * H.MAXSEQ, dtype=np.uint64); nseq = np.zeros(nblk, dtype=np.uint32)
        pP = np.zeros(NP, dtype=np.uint16); cP = np.zeros(5, dtype=np.uint32); pR = np.zeros(NP, dtype=np.uint16); cR = np.zeros(5, dtype=np.uint32)
        O.b2zo_lzma2_parse_final_model(src.ctypes.data, n, ctypes.byref(p), seqs.ctypes.data, nseq.ctypes.data, pP.ctypes.data, cP.ctypes.data)
        resets = O.b2zo_lzma2_final_model(src.ctypes.data, n, ctypes.byref(p), seqs.ctypes.data, nseq.ctypes.data, pR.ctypes.data, cR.ctypes.data)
        slice_bytes = (1 << fl) >> sl
        assert resets == (n + slice_bytes - 1) // slice_bytes        # no raw-chunk fallback reset the coder's model on the way
        assert np.array_equal(cP, cR) and np.array_equal(pP, pR)
        assert int((pP != 1024).sum()) > 500                          # and it is a model that has adapted
