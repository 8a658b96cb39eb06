"""CPU tests: pin the oracle (a) against the reference's golden vector, (b) against the
reference itself compiled from /root/reference (oracle/_ref) when present, and check the
encoder restatement round-trips through both decoders."""
import hashlib
import os

import pytest

import helpers

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def test_decoder_golden_reference_vector():
    """tests/regr-arc/test.txt.zstd of the reference (67 B, checksum flag set): payload SHA-256 is the
    one the reference's regression.test expects."""
    comp = open(os.path.join(GOLDEN, "test.txt.zstd"), "rb").read()
    out = helpers.oracle_decompress(comp, 1_000_000)
    assert len(out) == 1_000_000
    assert out == b"TEST\n" + b" " * 999990 + b"\nEND."
    assert hashlib.sha256(out).hexdigest() == open(os.path.join(GOLDEN, "test.txt.sha256")).read().strip()


def test_decoder_golden_frames():
    """frames produced by the reference encoder in this container (tests/golden/make_golden.py)."""
    import json
    idx = json.load(open(os.path.join(GOLDEN, "frames.json")))
    for name, meta in idx.items():
        comp = open(os.path.join(GOLDEN, name), "rb").read()
        out = helpers.oracle_decompress(comp, meta["size"])
        assert hashlib.sha256(out).hexdigest() == meta["sha256"], name


def test_xxh64_known_answers():
    import ctypes
    O = helpers.oracle()
    # published XXH64 test vectors (seed 0): empty input, and "a"
    assert O.b2zo_xxh64(None, 0, 0) == 0xEF46DB3751D8E999
    b = ctypes.create_string_buffer(b"a")
    assert O.b2zo_xxh64(b, 1, 0) == 0xD24EC4F1A98C6E5B


@pytest.mark.skipif(not helpers.ref_available(), reason="oracle/_ref not built (needs /root/reference)")
def test_decoder_vs_reference_encoder(pkg):
    datas = helpers.sample_inputs(pkg)
    for name, d in datas.items():
        for lv in (-5, 1, 3, 6, 13, 19):
            for cs in (0, 1):
                if len(d) > 500_000 and lv > 6:
                    continue
                comp = helpers.ref_compress(d, lv, cs)
                assert helpers.oracle_decompress(comp, len(d)) == d, (name, lv, cs)
    d = datas["g2_1m"]
    multi = helpers.ref_compress(d, 3) + b"\x50\x2a\x4d\x18\x04\x00\x00\x00ABCD" + helpers.ref_compress(datas["mixed"], 5, 1) + helpers.ref_compress(b"", 3)
    assert helpers.oracle_decompress(multi, len(d) + len(datas["mixed"])) == d + datas["mixed"]
    mt = helpers.ref_compress(d + d, 3, 0, nbWorkers=2)
    assert helpers.oracle_decompress(mt, 2 * len(d)) == d + d


def test_decoder_rejects_corruption(pkg):
    import random
    d = helpers.sample_inputs(pkg)["g2_100k"]
    comp = bytearray(helpers.oracle_compress(d))
    rnd = random.Random(7)
    undetected = 0
    for _ in range(200):
        c2 = bytearray(comp); i = rnd.randrange(len(c2)); c2[i] ^= 1 << rnd.randrange(8)
        try:
            if helpers.oracle_decompress(bytes(c2), len(d) + 64) == d:
                undetected += 1
        except ValueError:
            pass
    assert undetected == 0


def test_encoder_restatement_roundtrips(pkg):
    for name, d in helpers.sample_inputs(pkg, big=True).items():
        comp = helpers.oracle_compress(d)
        assert helpers.oracle_decompress(comp, len(d)) == d, name
        assert helpers.ref_zstd_result(comp, len(d)) == helpers.digest(d), name
    d = helpers.sample_inputs(pkg)["mixed"]
    for kw in (dict(frameLog=17, windowLog=17), dict(frameLog=20, windowLog=18, hashLogL=14, hashLogS=12), dict(flags=1)):
        comp = helpers.oracle_compress(d, **kw)
        assert helpers.oracle_decompress(comp, len(d)) == d, kw
        assert helpers.ref_zstd_result(comp, len(d)) == helpers.digest(d), kw


def test_encoder_ratio_vs_reference(pkg):
    d = pkg.corpus.g2(8 << 20).tobytes()
    ours = len(helpers.oracle_compress(d)); ref = helpers.ref_size(helpers.ref_compress, d, 3)
    assert ours <= ref * 1.01, (ours, ref)


def test_reference_regression_archives():
    """Packed streams of the reference's own regression archives (tests/regr-arc/*.7z -> tests/golden/regr_*, see
    make_golden_regr.py): level 17, ZSTD:max and solid folders; payload SHA-256 as regression.test expects."""
    import hashlib, json
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    idx = json.load(open(os.path.join(gold, "regr.json")))
    seen = 0
    for name, meta in idx.items():
        comp = open(os.path.join(gold, name), "rb").read()
        if meta["method"] == "zstd":
            out = helpers.oracle_decompress(comp, meta["size"])
        else:
            out, used = helpers.oracle_lzma2_decompress(comp, meta["size"], meta["dict_prop"]); assert used == len(comp)
        assert len(out) == meta["size"] and hashlib.sha256(out).hexdigest() == meta["sha256"], name
        seen += 1
    assert seen == 4
