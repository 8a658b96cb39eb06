"""CPU: oracle/lzma2_enc_oracle.c (the sequential statement of the GPU LZMA2 encoder) writes valid LZMA2: the reference
decoder (oracle/_ref, C/Lzma2Dec.c), liblzma and the oracle decoder all restore the input; block structure and ratio sanity."""
import lzma

import pytest

import helpers as H


def _dict_size(prop):
    return (2 | (prop & 1)) << (prop // 2 + 11)


def test_roundtrip_three_decoders(pkg):
    for name, data in H.sample_inputs(pkg, big=True).items():
        prop, comp = H.oracle_lzma2_compress(data)
        assert prop == 16 and comp[-1] == 0
        assert H.oracle_lzma2_decompress(comp, len(data), prop) == (data, len(comp)), name
        assert lzma.LZMADecompressor(format=lzma.FORMAT_RAW, filters=[{"id": lzma.FILTER_LZMA2, "dict_size": _dict_size(prop)}]).decompress(comp) == data, name
        assert H.ref_lzma2_result(comp, len(data), prop) == (H.digest(data), len(comp)), name


def test_frame_geometry_and_ratio(pkg):
    data = pkg.corpus.g2(3 * (1 << 20) + 12345).tobytes()
    for fl in (17, 18, 20):
        prop, comp = H.oracle_lzma2_compress(data, frameLog=fl, windowLog=fl)
        assert prop == (fl - 12) * 2
        out, used = H.oracle_lzma2_decompress(comp, len(data), prop)
        assert out == data and used == len(comp)
        nreset = 0; ip = 0                                        # every frame starts with a dictionary reset
        while comp[ip] != 0:
            ctl = comp[ip]
            if ctl == 1 or ctl >= 0xE0:
                nreset += 1
            if ctl <= 2:
                ip += 3 + ((comp[ip + 1] << 8) | comp[ip + 2]) + 1
            else:
                ip += 5 + (1 if ctl >= 0xC0 else 0) + ((comp[ip + 3] << 8) | comp[ip + 4]) + 1
        assert nreset == (len(data) + (1 << fl) - 1) >> fl
    prop, comp = H.oracle_lzma2_compress(data)
    zs = H.oracle_compress(data)
    assert len(comp) < len(zs) * 1.01                             # the same parse (priced for the zstd codes by stage G), range-coded: within 1 % of the zstd frames
    fl2 = H.ref_size(H.ref_fl2_compress, data, 5)
    assert len(comp) < 1.15 * fl2                        # greedy level-3-class parse in 1 MiB blocks vs FL2 level 5 (optimal parse, 8 MiB dictionary)


def test_incompressible_and_chunk_rollover(pkg):
    noise = pkg.corpus.entropy_class(1, 400_000).tobytes()
    prop, comp = H.oracle_lzma2_compress(noise)
    assert len(comp) <= len(noise) + 3 * (len(noise) // 60000 + 2) + 1      # raw-chunk fallback
    assert H.oracle_lzma2_decompress(comp, len(noise), prop)[0] == noise
    mixed = noise[:100_000] + bytes(300_000) + pkg.corpus.g2(500_000).tobytes() + noise[100_000:200_000]
    prop, comp = H.oracle_lzma2_compress(mixed)
    assert H.oracle_lzma2_decompress(comp, len(mixed), prop)[0] == mixed
    assert H.ref_lzma2_result(comp, len(mixed), prop)[0] == H.digest(mixed)


def test_state_reset_slices(pkg):
    """flags bits 8..10: a block's range coding split into state-reset slices (independent chains for the GPU): still one
    dictionary-reset block per frame, every decoder restores the input, and the ratio cost stays small."""
    data = pkg.corpus.g2(2 * (1 << 20) + 300_000).tobytes() + pkg.corpus.entropy_class(1, 200_000).tobytes()
    sizes = []
    for sl in range(4):
        prop, comp = H.oracle_lzma2_compress(data, flags=1 | (sl << 8))
        assert H.oracle_lzma2_decompress(comp, len(data), prop) == (data, len(comp))
        assert lzma.LZMADecompressor(format=lzma.FORMAT_RAW, filters=[{"id": lzma.FILTER_LZMA2, "dict_size": _dict_size(prop)}]).decompress(comp) == data
        assert H.ref_lzma2_result(comp, len(data), prop) == (H.digest(data), len(comp))
        assert H.ref_lzma2_mt_result(comp, len(data), prop, 4) == (H.digest(data), True)
        sizes.append(len(comp))
    assert sizes[0] <= sizes[1] <= sizes[2] <= sizes[3] < sizes[0] * 1.01


def test_large_frames_hit_the_unpack_limit(pkg):
    """Frames of 2..16 MiB with very compressible data: chunks close at the 2 MiB - 512 unpack limit, not the pack limit."""
    data = pkg.corpus.entropy_class(3, 5 << 20).tobytes() + bytes(4 << 20)
    for fl, sl in ((21, 0), (23, 2), (24, 0)):
        prop, comp = H.oracle_lzma2_compress(data, frameLog=fl, windowLog=fl, flags=1 | (sl << 8))
        assert prop == (fl - 12) * 2
        assert H.oracle_lzma2_decompress(comp, len(data), prop) == (data, len(comp))
        assert H.ref_lzma2_result(comp, len(data), prop) == (H.digest(data), len(comp))
