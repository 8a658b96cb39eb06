"""GPU parity tests of stage Z, the price-based Zstandard parse (B200Z_P_ZSTD_PARSE = 1 / B200Z_P_LEVEL >= 8; csrc/zstd_enc_parse.cu on
stage C's candidates) through the C ABI: sequences and literals must equal the oracle's (oracle/zstd_opt_oracle.c), frames must
equal the oracle's byte for byte, and the reference decoder / our GPU decoder must restore the input.

Sorts last on purpose: this kernel was written after the round's GPU budget was spent.  Its logic is checked against the oracle
through the host emulation of the kernel source (tests/test_cuemu_kernels.py), as stage C / stage P were before their first
(passing) hardware run; the first hardware run of stage Z is the one that happens here."""
import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu
ZOPT = 0x20


@pytest.fixture(scope="module")
def inputs(pkg):
    return helpers.sample_inputs(pkg, big=False)


@pytest.fixture(scope="module")
def zcodec(pkg):
    c = pkg.Codec(0, zstd_parse=1)
    yield c
    c.close()


def test_stage_tap_equals_the_oracle(pkg, inputs):
    for fl in (20, 18):
        c = pkg.Codec(0, frame_log=fl, window_log=fl, zstd_parse=1)
        for name, data in inputs.items():
            if not data:
                continue
            seqs, nseq, lits, nlit = c.stage_m(data)
            ws, wn, wl, wnl = helpers.oracle_find_sequences(data, frameLog=fl, windowLog=fl, flags=1 | ZOPT)
            assert np.array_equal(nseq, wn) and np.array_equal(nlit, wnl), (name, fl)
            for b in range(len(wn)):
                assert np.array_equal(seqs[b * helpers.MAXSEQ:b * helpers.MAXSEQ + wn[b]], ws[b * helpers.MAXSEQ:b * helpers.MAXSEQ + wn[b]]), (name, fl, b)
                assert np.array_equal(lits[b * 131072:b * 131072 + wnl[b]], wl[b * 131072:b * 131072 + wnl[b]]), (name, fl, b)
        c.close()


def test_frames_bit_exact_and_decoders_accept(zcodec, inputs):
    for name, data in inputs.items():
        comp = zcodec.compress(data)
        assert comp == helpers.oracle_compress(data, flags=1 | ZOPT), name
        assert helpers.oracle_decompress(comp, len(data)) == data, name
        assert helpers.ref_zstd_result(comp, len(data)) == helpers.digest(data), name
        assert zcodec.decompress(comp) == data, name


def test_level_selects_the_parse_and_checksums(pkg, inputs):
    data = inputs["mixed"] + inputs["g2_1m"]
    want = helpers.oracle_compress(data, flags=1 | ZOPT)
    for level in (8, 19):
        c = pkg.Codec(0, level=level)
        assert c.get("zstd_parse") == 1 and c.compress(data) == want
        c.close()
    c = pkg.Codec(0, level=4)                                    # (levels 3-4: the oracle's default parameters; the other rungs: test_level_ladder_matches_oracle)
    assert c.get("zstd_parse") == 0 and c.compress(data) == helpers.oracle_compress(data)
    c.close()
    c = pkg.Codec(0, level=12, flags=3)                          # + XXH64 content checksum
    comp = c.compress(data)
    assert comp == helpers.oracle_compress(data, flags=3 | ZOPT) and c.decompress(comp) == data
    c.close()


def test_codec_module_level_selects_the_parse(pkg, tmp_path):
    """ICompressCoder::Code() of the ZSTD coder class at level 12 (kLevel -> B200Z_P_LEVEL >= 8): stage Z's frames, accepted by the reference decoder"""
    import os
    import subprocess
    PKG = os.path.join(helpers.ROOT, "7-zip-zstd_b200")
    data = pkg.corpus.g2(5 * (1 << 20) + 999).tobytes() + bytes(300000)
    src = tmp_path / "in.bin"; packed = tmp_path / "packed.zst"
    src.write_bytes(data)
    out = subprocess.run([os.path.join(PKG, "build", "coder_roundtrip"), os.path.join(PKG, "libb200z_7z.so"), str(src), str(packed), "12"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "roundtrip ok" in out.stdout, out.stderr + out.stdout
    comp = packed.read_bytes()
    assert comp == helpers.oracle_compress(data, flags=1 | ZOPT)
    assert helpers.ref_zstd_result(comp, len(data)) == helpers.digest(data)


def test_sequence_array_full(pkg, zcodec):
    """random 3-byte tokens: a block wants more than 32 768 sequences; the rule for the overflow and the 3-byte sequence-count form"""
    import random
    rng = random.Random(1)
    toks = [bytes(rng.randrange(256) for _ in range(3)) for _ in range(64)]
    data = b"".join(rng.choice(toks) for _ in range(500_000))[:(1 << 20) + 5000]
    assert int(helpers.oracle_find_sequences(data, flags=1 | ZOPT)[1].max()) == helpers.MAXSEQ
    comp = zcodec.compress(data)
    assert comp == helpers.oracle_compress(data, flags=1 | ZOPT)
    assert zcodec.decompress(comp) == data
    assert helpers.ref_zstd_result(comp, len(data)) == helpers.digest(data)


def test_capped_candidate_is_clipped_at_a_block_end(pkg, zcodec):
    data = helpers.capped_match_near_boundary(pkg)
    comp = zcodec.compress(data)
    assert comp == helpers.oracle_compress(data, flags=1 | ZOPT)
    assert zcodec.decompress(comp) == data


def test_large_frames_batches_and_ratio(pkg):
    data = pkg.corpus.g2(9 * (1 << 20) + 4321).tobytes()
    c = pkg.Codec(0, frame_log=22, window_log=22, zstd_parse=1)
    comp = c.compress(data)
    assert comp == helpers.oracle_compress(data, frameLog=22, windowLog=22, flags=1 | ZOPT)
    assert c.decompress(comp) == data
    c.close()
    l3 = pkg.Codec(0); g = l3.compress(data); l3.close()
    assert len(comp) < 0.94 * len(g)                              # measured on the oracle: 2.60 against 2.39
    import torch
    c = pkg.Codec(0, batch_log=22, zstd_parse=1)                  # device-pointer entry, several kernel batches
    d_src = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    cap = c.compress_bound(len(data))
    d_dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    n = c.compress_device(d_src.data_ptr(), len(data), d_dst.data_ptr(), cap)
    assert d_dst[:n].cpu().numpy().tobytes() == helpers.oracle_compress(data, flags=1 | ZOPT)
    c.close()


def test_large_roundtrip_property(pkg):
    """size-independent property at a larger size: decode(encode(x)) == x through both GPU paths, many blocks"""
    data = pkg.corpus.g2(64 << 20, seed=79)
    c = pkg.Codec(0, level=16)
    comp = c.compress(data)
    out = c.decompress(comp)
    assert np.array_equal(np.frombuffer(out, dtype=np.uint8), data)
    assert data.nbytes / len(comp) > 2.45           # 2.54 on this seed (oracle); stage M: 2.39
    c.close()
