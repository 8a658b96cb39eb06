"""GPU parity tests of the LZMA2 encoder through the C ABI: the stream must equal the oracle's byte for byte (stage M is
shared with the zstd path, stage R is oracle/lzma2_enc_oracle.c), and the reference decoder / liblzma / our GPU decoder
must restore the input from it."""
import lzma

import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu


def _dict_size(prop):
    return (2 | (prop & 1)) << (prop // 2 + 11)


@pytest.fixture(scope="module")
def inputs(pkg):
    return helpers.sample_inputs(pkg, big=True)


def test_bit_exact_vs_oracle(codec, inputs):
    for name, data in inputs.items():
        prop, comp = codec.lzma2_compress(data)
        oprop, want = helpers.oracle_lzma2_compress(data)
        assert prop == oprop and comp == want, name


def test_decoders_accept(codec, inputs):
    for name, data in inputs.items():
        prop, comp = codec.lzma2_compress(data)
        assert lzma.LZMADecompressor(format=lzma.FORMAT_RAW, filters=[{"id": lzma.FILTER_LZMA2, "dict_size": _dict_size(prop)}]).decompress(comp) == data, name
        assert helpers.ref_lzma2_result(comp, len(data), prop) == (helpers.digest(data), len(comp)), name
        assert codec.lzma2_decompress(comp, prop) == data, name
        size, nblk, used = codec.lzma2_stream_info(comp)
        assert size == len(data) and used == len(comp) and nblk == (len(data) + (1 << 20) - 1) >> 20


def test_geometry_model_placement_and_batches(pkg, inputs):
    data = inputs["g2_9m"]
    want = {fl: helpers.oracle_lzma2_compress(data, frameLog=fl, windowLog=fl) for fl in (17, 20)}
    for fl in (17, 20):
        for model in (1, 2, 3):                            # literal model in shared / global memory (one chain per warp), 3 = 32 chains per warp in lock-step
            c = pkg.Codec(0, frame_log=fl, window_log=fl, lzma2_model=model)
            assert c.lzma2_compress(data) == want[fl], (fl, model)
            c.close()
    for sl in (0, 1, 3):                                    # state-reset slices per block (default 2 is what every other test runs)
        c = pkg.Codec(0, lzma2_slice_log=sl)
        assert c.lzma2_compress(data) == helpers.oracle_lzma2_compress(data, flags=1 | (sl << 8)), sl
        c.close()
    # device-pointer entry with several kernel batches: same bytes (every batch's end marker is overwritten by the next)
    import torch
    c = pkg.Codec(0, batch_log=22)
    d_src = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    cap = c.lzma2_compress_bound(len(data))
    d_dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    n, prop = c.lzma2_compress_device(d_src.data_ptr(), len(data), d_dst.data_ptr(), cap)
    assert (prop, d_dst[:n].cpu().numpy().tobytes()) == want[20]
    c.close()


def test_large_roundtrip_property(codec, pkg):
    """size-independent property at a larger size: decode(encode(x)) == x through both GPU paths, many blocks"""
    data = pkg.corpus.g2(96 << 20, seed=77)
    prop, comp = codec.lzma2_compress(data)
    assert codec.lzma2_stream_info(comp)[1] == 96
    out = codec.lzma2_decompress(comp, prop)
    assert np.array_equal(np.frombuffer(out, dtype=np.uint8), data)


def test_device_count_is_invisible(pkg):
    """method 21 through a context over several workers (every GPU of the box; one GPU listed twice where there is only one):
    batches of whole dictionary-reset blocks are dealt over them and stitched without end markers in between -- the chunk stream
    equals the single-device / oracle stream"""
    import torch
    data = pkg.corpus.g2(40 * (1 << 20) + 4321).tobytes()
    oprop, want = helpers.oracle_lzma2_compress(data, frameLog=17, windowLog=17)
    n = torch.cuda.device_count()
    for devs in ([0, 0], list(range(n)) if n >= 2 else [0, 0, 0]):
        c = pkg.Codec(devices=devs, frame_log=17)
        prop, comp = c.lzma2_compress(data)
        assert prop == oprop and comp == want, devs
        assert c.lzma2_decompress(comp, prop) == data
        c.close()
