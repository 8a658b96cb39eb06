"""GPU parity tests of the price-based parse of the method-21 encoder (B200Z_P_LZMA2_PARSE = 1; csrc/lzma2_parse.cu) through the
C ABI: stage C's candidate words and stage P's sequences must equal the oracle's (oracle/lzma2_opt_oracle.c), the final stream
must equal the oracle's byte for byte, and the reference decoder / liblzma / our GPU decoder must restore the input.

This file sorts after the other GPU tests on purpose: these kernels were written in a session whose GPU budget was spent, so
their logic has been checked against the oracle through the host emulation of the kernel sources (tests/test_cuemu_kernels.py)
but the first run on hardware is the one that happens here."""
import ctypes
import lzma

import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu
OPT = 0x10


def _dict_size(prop):
    return (2 | (prop & 1)) << (prop // 2 + 11)


def _oracle_taps(data, fl, flags):
    O = helpers.oracle()
    O.b2zo_lzma2_candidates.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p]
    O.b2zo_lzma2_parse_frame.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.POINTER(helpers.EncParams)] + [ctypes.c_void_p] * 3
    n = len(data); F = 1 << fl; bpf = F >> 17
    src = np.frombuffer(data, dtype=np.uint8)
    nblk = (n + 131071) // 131072
    cand = np.zeros(n * 4, dtype=np.uint32); seqs = np.zeros(nblk * helpers.MAXSEQ, dtype=np.uint64); nseq = np.zeros(nblk, dtype=np.uint32)
    p = helpers.enc_params(frameLog=fl, windowLog=fl, flags=flags)
    for f0 in range(0, n, F):
        fn = min(F, n - f0); b0 = (f0 // F) * bpf
        O.b2zo_lzma2_candidates(src.ctypes.data + f0, fn, fl, cand.ctypes.data + f0 * 16)
        O.b2zo_lzma2_parse_frame(src.ctypes.data + f0, fn, ctypes.byref(p), cand.ctypes.data + f0 * 16, seqs.ctypes.data + b0 * helpers.MAXSEQ * 8, nseq.ctypes.data + b0 * 4)
    return cand.reshape(-1, 4), seqs, nseq


@pytest.fixture(scope="module")
def inputs(pkg):
    return helpers.sample_inputs(pkg, big=False)


@pytest.fixture(scope="module")
def opt_codec(pkg):
    c = pkg.Codec(0, lzma2_parse=1)
    yield c
    c.close()


def test_stage_taps_equal_the_oracle(pkg, inputs):
    for fl, sl in ((20, 2), (18, 0)):
        c = pkg.Codec(0, frame_log=fl, window_log=fl, lzma2_slice_log=sl, lzma2_parse=1)
        for name, data in inputs.items():
            if not data:
                continue
            cand, seqs, nseq = c.stage_cp(data)
            wc, ws, wn = _oracle_taps(data, fl, 1 | (sl << 8) | OPT)
            assert np.array_equal(cand, wc), (name, fl, "stage C")
            assert np.array_equal(nseq, wn), (name, fl, "stage P counts")
            for b in range(len(wn)):
                assert np.array_equal(seqs[b * helpers.MAXSEQ:b * helpers.MAXSEQ + wn[b]], ws[b * helpers.MAXSEQ:b * helpers.MAXSEQ + wn[b]]), (name, fl, b)
        c.close()


def test_stream_bit_exact_and_decoders_accept(opt_codec, inputs):
    for name, data in inputs.items():
        prop, comp = opt_codec.lzma2_compress(data)
        assert (prop, comp) == helpers.oracle_lzma2_compress(data, flags=1 | (2 << 8) | OPT), name
        assert lzma.LZMADecompressor(format=lzma.FORMAT_RAW, filters=[{"id": lzma.FILTER_LZMA2, "dict_size": _dict_size(prop)}]).decompress(comp) == data, name
        assert helpers.ref_lzma2_result(comp, len(data), prop) == (helpers.digest(data), len(comp)), name
        assert opt_codec.lzma2_decompress(comp, prop) == data, name


def test_large_frames_batches_and_ratio(pkg):
    data = pkg.corpus.g2(9 * (1 << 20) + 4321).tobytes()
    c = pkg.Codec(0, frame_log=22, window_log=22, lzma2_slice_log=3, lzma2_parse=1)
    prop, comp = c.lzma2_compress(data)
    assert (prop, comp) == helpers.oracle_lzma2_compress(data, frameLog=22, windowLog=22, flags=1 | (3 << 8) | OPT)
    assert c.lzma2_decompress(comp, prop) == data
    c.close()
    greedy = pkg.Codec(0); g = greedy.lzma2_compress(data)[1]; greedy.close()
    assert len(comp) < 0.93 * len(g)                              # measured on the oracle: 2.62 against 2.40
    # device-pointer entry, several kernel batches: same bytes as one batch
    import torch
    c = pkg.Codec(0, batch_log=22, lzma2_parse=1)
    d_src = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    cap = c.lzma2_compress_bound(len(data))
    d_dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    n, prop = c.lzma2_compress_device(d_src.data_ptr(), len(data), d_dst.data_ptr(), cap)
    assert (prop, d_dst[:n].cpu().numpy().tobytes()) == helpers.oracle_lzma2_compress(data, flags=1 | (2 << 8) | OPT)
    c.close()


@pytest.mark.parametrize("method,level", [("lzma2", 5), ("flzma2", 5), ("flzma2", 3)])
def test_codec_module_selects_the_price_based_parse(pkg, tmp_path, method, level):
    from test_boundary import codec_module_lzma2_roundtrip
    codec_module_lzma2_roundtrip(pkg, tmp_path, method, level, True)


def test_capped_candidate_is_clipped_at_a_slice_end(pkg):
    """the case the emulator fuzz found after the first hardware run (helpers.capped_match_near_boundary)"""
    data = helpers.capped_match_near_boundary(pkg)
    c = pkg.Codec(0, frame_log=18, window_log=18, lzma2_slice_log=1, lzma2_parse=1)
    prop, comp = c.lzma2_compress(data)
    assert (prop, comp) == helpers.oracle_lzma2_compress(data, frameLog=18, windowLog=18, flags=1 | (1 << 8) | OPT)
    assert c.lzma2_decompress(comp, prop) == data
    assert helpers.ref_lzma2_result(comp, len(data), prop)[0] == helpers.digest(data)
    c.close()


def test_large_roundtrip_property(pkg):
    """size-independent property at a larger size: decode(encode(x)) == x through both GPU paths, many blocks"""
    data = pkg.corpus.g2(64 << 20, seed=78)
    c = pkg.Codec(0, lzma2_parse=1)
    prop, comp = c.lzma2_compress(data)
    out = c.lzma2_decompress(comp, prop)
    assert np.array_equal(np.frombuffer(out, dtype=np.uint8), data)
    assert len(data) / len(comp) > 2.45          # 2.50 on this seed (oracle); greedy: 2.36
    c.close()
