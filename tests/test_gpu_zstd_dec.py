"""GPU parity tests of the zstd decoder path (through the C ABI): output must be bit-exact
against the reference for any valid frame -- checked on frames produced by the reference encoder
(oracle/_ref) at many levels, on the committed golden fixtures (reference test vector + reference
encoder outputs), on our own encoder's frames, and on corrupted inputs against the oracle decoder."""
import hashlib
import json
import os
import random

import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def inputs(pkg):
    return helpers.sample_inputs(pkg, big=True)


def test_golden_reference_vector(codec):
    comp = open(os.path.join(GOLDEN, "test.txt.zstd"), "rb").read()
    out = codec.decompress(comp, max_size=1_000_000)      # the vector declares no content size
    assert hashlib.sha256(out).hexdigest() == open(os.path.join(GOLDEN, "test.txt.sha256")).read().strip()


def test_golden_reference_frames(codec):
    idx = json.load(open(os.path.join(GOLDEN, "frames.json")))
    for name, meta in idx.items():
        comp = open(os.path.join(GOLDEN, name), "rb").read()
        out = codec.decompress(comp, max_size=meta["size"])
        assert hashlib.sha256(out).hexdigest() == meta["sha256"], name


def test_own_frames_roundtrip(codec, inputs):
    for name, data in inputs.items():
        comp = codec.compress(data)
        assert codec.decompress(comp) == data, name


@pytest.mark.skipif(not helpers.ref_available(), reason="oracle/_ref not built")
def test_reference_encoder_frames(codec, inputs):
    for name, d in inputs.items():
        for lv in (-5, 1, 3, 6, 13, 19):
            for cs in (0, 1):
                if len(d) > 1_100_000 and lv > 6:
                    continue
                comp = helpers.ref_compress(d, lv, cs)
                assert codec.decompress(comp, max_size=len(d)) == d, (name, lv, cs)
    d = inputs["g2_1m"]
    multi = helpers.ref_compress(d, 3) + b"\x50\x2a\x4d\x18\x04\x00\x00\x00ABCD" + helpers.ref_compress(inputs["mixed"], 5, 1) + helpers.ref_compress(b"", 3)
    assert codec.decompress(multi, max_size=len(d) + len(inputs["mixed"])) == d + inputs["mixed"]
    mt = helpers.ref_compress(d + d, 3, 0, nbWorkers=2)                 # zstdmt: one frame, jobs without frame headers
    assert codec.decompress(mt, max_size=2 * len(d)) == d + d
    nofcs = helpers.ref_compress(inputs["mixed"], 4, 0, contentSizeFlag=0)     # streaming-style frame: no content size
    assert codec.decompress(nofcs, max_size=len(inputs["mixed"])) == inputs["mixed"]


def test_corrupted_inputs_match_oracle(pkg, codec, inputs):
    """bit flips: the GPU decoder must fail cleanly or produce exactly what the oracle decoder produces"""
    d = inputs["mixed"][:300_000]
    comp = bytearray(codec.compress(d))
    rnd = random.Random(11)
    for _ in range(40):
        c2 = bytearray(comp)
        for _k in range(rnd.randrange(1, 3)):
            i = rnd.randrange(len(c2)); c2[i] ^= 1 << rnd.randrange(8)
        try:
            want = helpers.oracle_decompress(bytes(c2), len(d) + 4096)
        except ValueError:
            want = None
        try:
            got = codec.decompress(bytes(c2), max_size=len(d) + 4096)
        except pkg.B200zError:
            got = None
        assert got == want
    with pytest.raises(pkg.B200zError):
        codec.decompress(b"not a zstd frame at all", max_size=100)
    with pytest.raises(pkg.B200zError):
        codec.decompress(bytes(comp[: len(comp) // 2]), max_size=len(d))


def test_dst_too_small(pkg, codec, inputs):
    comp = codec.compress(inputs["g2_1m"])
    with pytest.raises(pkg.B200zError) as e:
        codec.decompress(comp, max_size=1000)
    assert e.value.code == -4


def test_device_resident_decode(pkg, codec):
    import torch
    data = pkg.corpus.g2(8 << 20)
    comp = np.frombuffer(codec.compress(data.tobytes()), dtype=np.uint8)
    src = torch.from_numpy(comp.copy()).cuda()
    dst = torch.empty(data.size, dtype=torch.uint8, device="cuda")
    codec.reset_stats()
    n = codec.decompress_device(src.data_ptr(), src.numel(), dst.data_ptr(), dst.numel())
    assert n == data.size and bytes(dst.cpu().numpy()) == data.tobytes()
    assert codec.stat(4) > 0 and codec.stat(5) > 0


def test_host_pipeline_batches(pkg):
    """the H2D | kernels | D2H pipeline of the host-pointer entry points (many small batches) gives the same bytes"""
    data = pkg.corpus.g2(37 * (1 << 20) + 4567).tobytes()
    c = pkg.Codec(0, host_batch_log=22)
    comp = c.compress(data)
    assert comp == helpers.oracle_compress(data)
    assert c.decompress(comp) == data
    c.close()


def test_content_checksums(pkg, inputs):
    """flag bit1: frames carry XXH64 checksums -- same bytes as the oracle, accepted by the reference decoder
    (which verifies them), verified by the GPU decoder, and a flipped checksum is reported as such."""
    data = inputs["mixed"] + inputs["g2_1m"][:777_777]
    c = pkg.Codec(0, flags=3)
    comp = c.compress(data)
    assert comp == helpers.oracle_compress(data, flags=3)
    assert c.compress(b"") == helpers.oracle_compress(b"", flags=3)
    assert helpers.ref_zstd_result(comp, len(data)) == helpers.digest(data)
    assert helpers.ref_zstd_result(c.compress(b""), 0) == helpers.digest(b"")
    assert c.decompress(comp) == data
    bad = bytearray(comp); bad[-1] ^= 0x40                                   # last byte = part of the last frame's checksum
    with pytest.raises(pkg.B200zError) as e:
        c.decompress(bytes(bad), max_size=len(data))
    assert e.value.code == -8
    if helpers.ref_available():                                               # reference-made frames with checksums at odd output offsets
        a, b = inputs["g2_100k"][:99_999], inputs["tile"][:123_457]
        two = helpers.ref_compress(a, 3, 1) + helpers.ref_compress(b, 5, 1)
        assert c.decompress(two, max_size=len(a) + len(b)) == a + b
        bad = bytearray(two); bad[len(helpers.ref_compress(a, 3, 1)) - 2] ^= 1
        with pytest.raises(pkg.B200zError) as e:
            c.decompress(bytes(bad), max_size=len(a) + len(b))
        assert e.value.code == -8
    c.close()


def test_reference_regression_archives(codec):
    """Packed streams of the reference's own regression archives (tests/regr-arc/*.7z): both methods, solid folders, ZSTD:max."""
    idx = json.load(open(os.path.join(GOLDEN, "regr.json")))
    for name, meta in idx.items():
        comp = open(os.path.join(GOLDEN, name), "rb").read()
        out = codec.decompress(comp, max_size=meta["size"]) if meta["method"] == "zstd" else codec.lzma2_decompress(comp, meta["dict_prop"])
        assert len(out) == meta["size"] and hashlib.sha256(out).hexdigest() == meta["sha256"], name


@pytest.mark.skipif(not helpers.ref_available(), reason="oracle/_ref not built")
def test_stage_j_pointer_jumping(pkg, inputs):
    """stage J on hardware: forced on every frame (mode 2) it restores what the execution units restore -- reference frames of several
    levels, frames with raw / RLE blocks and long runs, several frames in one call, a damaged stream (same verdict as the oracle decoder);
    in automatic mode a reference-written 48 MiB frame (sliding window: its units would run one behind the other) is taken by stage J, a
    long-mode frame of this encoder (independent regions) and the short frames are not; host batches and the device-pointer call agree"""
    S_JUMP = 11
    off, auto, force = pkg.Codec(0, dec_jump=0), pkg.Codec(0), pkg.Codec(0, dec_jump=2)
    for name, d in inputs.items():
        for comp in (helpers.ref_compress(d, 3), helpers.ref_compress(d, 19 if len(d) < 600_000 else 5, 1), off.compress(d)):
            force.reset_stats()
            assert force.decompress(comp, max_size=len(d)) == d, name
            assert force.stat(S_JUMP) > 0 or not d, name
            assert off.decompress(comp, max_size=len(d)) == d and off.stat(S_JUMP) == 0
    d = inputs["mixed"]
    comp = helpers.ref_compress(d, 4)
    for pos in (len(comp) // 3, len(comp) // 2, len(comp) - 9):
        bad = bytearray(comp); bad[pos] ^= 0x41
        try:
            want = helpers.oracle_decompress(bytes(bad), len(d))
        except ValueError:
            want = None
        try:
            got = force.decompress(bytes(bad), max_size=len(d))
        except pkg.B200zError:
            got = None
        assert got == want, pos
    big = helpers.far_copies(pkg, 48 << 20, every=1 << 22, span=(100_000, 900_000), seed=5) + bytes(1 << 20) + b"ab" * 300_000
    ref = helpers.ref_compress(big, 3, 0, nbWorkers=4)
    for c, jumped in ((auto, 1), (force, 1), (off, 0)):
        c.reset_stats()
        assert c.decompress(ref, max_size=len(big)) == big
        assert c.stat(S_JUMP) == jumped
    lng = pkg.Codec(0, long=24)
    ours = lng.compress(big); lng.close()
    auto.reset_stats()
    assert auto.decompress(ours) == big and auto.stat(S_JUMP) == 0
    multi = ref + off.compress(d) + ref
    auto.reset_stats()
    assert auto.decompress(multi, max_size=2 * len(big) + len(d)) == big + d + big and auto.stat(S_JUMP) == 2
    seg = pkg.Codec(0, dec_jump_seg_log=20)                             # the output resolved in 1 MiB segments, in order: blocks straddle the cuts
    assert seg.decompress(multi, max_size=2 * len(big) + len(d)) == big + d + big and seg.stat(S_JUMP) == 2
    seg.close()
    small = pkg.Codec(0, host_batch_log=24)                             # 16 MiB batches: every reference frame is a batch of its own
    assert small.decompress(multi, max_size=2 * len(big) + len(d)) == big + d + big and small.stat(S_JUMP) == 2
    for c in (off, auto, force, small):
        c.close()


@pytest.mark.skipif(not helpers.ref_available(), reason="oracle/_ref not built")
def test_stage_j_frame_beyond_2gib(pkg):
    """one reference-written frame of 2.5 GiB (zstdmt, level 1): stage J takes it in segments of 1 GiB -- pointers stay 31 bits whatever
    the frame's size -- and the output equals the input (compared on the device)"""
    import torch
    n = (5 << 29) + 12345
    data = pkg.corpus.g2(n)
    comp = helpers.ref_compress(data, 1, 0, nbWorkers=min(os.cpu_count() or 1, 64))
    c = pkg.Codec(0)
    src = torch.frombuffer(bytearray(comp + bytes(64)), dtype=torch.uint8).cuda()
    back = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
    got = c.decompress_device(src.data_ptr(), len(comp), back.data_ptr(), n)
    assert got == n and c.stat(11) == 1
    want = torch.from_numpy(data).cuda()
    assert bool(torch.equal(back[:n], want))
    c.close()
