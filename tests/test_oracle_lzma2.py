"""Pins oracle/lzma2_dec_oracle.c (CPU): golden LZMA2 streams from the reference's own regression archive, from the
reference's two encoders and from liblzma; plus agreement with the reference decoder when oracle/_ref is present."""
import hashlib
import json
import lzma
import os

import pytest

import helpers as H

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
IDX = json.load(open(os.path.join(GOLD, "lzma2.json")))


@pytest.mark.parametrize("name", sorted(IDX))
def test_golden_streams(name):
    meta = IDX[name]
    comp = open(os.path.join(GOLD, name), "rb").read()
    out, used = H.oracle_lzma2_decompress(comp, meta["size"], meta["dict_prop"])
    assert len(out) == meta["size"] and hashlib.sha256(out).hexdigest() == meta["sha256"]
    assert comp[used - 1] == 0 and used <= len(comp)          # stops on the end marker (FL2 appends a hash after it)
    assert H.ref_lzma2_result(comp, meta["size"], meta["dict_prop"]) == (H.digest(out), used)


def test_liblzma_streams(pkg):
    for seed, n, preset, lc, lp, pb in [(1, 50_000, 0, 3, 0, 2), (2, 200_000, 4, 0, 0, 0), (3, 90_000, 9, 4, 0, 4), (4, 3_000_000, 1, 1, 2, 3)]:
        data = pkg.corpus.g2(n, seed=seed).tobytes()
        comp = lzma.compress(data, format=lzma.FORMAT_RAW, filters=[dict(id=lzma.FILTER_LZMA2, preset=preset, dict_size=1 << 16, lc=lc, lp=lp, pb=pb)])
        out, used = H.oracle_lzma2_decompress(comp, n, 8)
        assert out == data and used == len(comp)


def test_errors():
    comp = open(os.path.join(GOLD, "lzma2_fl2_g2_100k.bin"), "rb").read()
    with pytest.raises(ValueError):
        H.oracle_lzma2_decompress(comp[:1000], 100_000, 10)              # truncated
    with pytest.raises(ValueError):
        H.oracle_lzma2_decompress(comp, 50_000, 10)                      # destination too small
    with pytest.raises(ValueError):
        H.oracle_lzma2_decompress(b"\x80" + comp[1:], 100_000, 10)       # first chunk without dictionary reset
    bad = bytearray(comp); bad[3000] ^= 0x55
    try:
        out, _ = H.oracle_lzma2_decompress(bytes(bad), 100_000, 10)      # corruption: an error or different bytes, never a crash
        assert hashlib.sha256(out).hexdigest() != IDX["lzma2_fl2_g2_100k.bin"]["sha256"]
    except ValueError:
        pass


def test_stream_info_host_walk():
    """b200z_lzma2_stream_info is host-only (chunk headers): sizes, block counts and malformed-stream detection, no GPU."""
    import ctypes
    lib = ctypes.CDLL(os.path.join(H.ROOT, "7-zip-zstd_b200", "libb200z.so"))
    lib.b200z_lzma2_stream_info.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_size_t)]
    for name, meta in IDX.items():
        comp = open(os.path.join(GOLD, name), "rb").read()
        buf = ctypes.create_string_buffer(comp, len(comp))
        cs, nb, used = ctypes.c_uint64(), ctypes.c_uint32(), ctypes.c_size_t()
        assert lib.b200z_lzma2_stream_info(buf, len(comp), ctypes.byref(cs), ctypes.byref(nb), ctypes.byref(used)) == 0
        assert cs.value == meta["size"] and comp[used.value - 1] == 0
        assert nb.value == (4 if name == "lzma2_lzma2_tile_blocks.bin" else (0 if meta["size"] == 0 else 1)), (name, nb.value)
        if len(comp) > 10:
            assert lib.b200z_lzma2_stream_info(buf, len(comp) // 2, ctypes.byref(cs), ctypes.byref(nb), ctypes.byref(used)) == -5


def test_corruption_parity_with_reference():
    """Bit flips and truncations: the oracle accepts exactly what the reference decoder (C/Lzma2Dec.c: Lzma2Decode) accepts,
    with the same bytes and the same consumed count -- the error behaviour the GPU decoder is then tested against."""
    import random
    rng = random.Random(3)
    accepted = 0
    for name, meta in IDX.items():
        comp = open(os.path.join(GOLD, name), "rb").read()
        if len(comp) < 50:
            continue
        for _ in range(60):
            bad = bytearray(comp); k = rng.randrange(len(comp)); bad[k] ^= 1 << rng.randrange(8)
            if rng.random() < 0.2:
                bad = bad[:rng.randrange(1, len(bad))]
            bad = bytes(bad)
            try:
                o = H.oracle_lzma2_decompress(bad, meta["size"], meta["dict_prop"])
            except ValueError:
                o = None
            assert H.lzma2_result(o) == H.ref_lzma2_result(bad, meta["size"], meta["dict_prop"]), (name, k)
            accepted += o is not None
    assert accepted > 10          # some corruptions are harmless (bytes after the end marker, FL2's trailing hash)


def test_chunk_header_rules_host_walk_and_oracle():
    """Lzma2Dec_UpdateState's needInitLevel rule and property checks (C/Lzma2Dec.c:97-165): the host walk
    (b200z_lzma2_stream_info) and the oracle decoder reject the same malformed chunk sequences."""
    import ctypes
    lib = ctypes.CDLL(os.path.join(H.ROOT, "7-zip-zstd_b200", "libb200z.so"))
    lib.b200z_lzma2_stream_info.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_size_t)]

    def walk(b):
        buf = ctypes.create_string_buffer(b, len(b)); cs, nb, used = ctypes.c_uint64(), ctypes.c_uint32(), ctypes.c_size_t()
        return lib.b200z_lzma2_stream_info(buf, len(b), ctypes.byref(cs), ctypes.byref(nb), ctypes.byref(used)), cs.value, nb.value, used.value

    raw = lambda ctl, payload: bytes([ctl, (len(payload) - 1) >> 8, (len(payload) - 1) & 0xFF]) + payload
    good = raw(1, b"hello") + raw(2, b" world") + b"\x00"
    assert walk(good) == (0, 11, 1, len(good)) and H.oracle_lzma2_decompress(good, 11, 0) == (b"hello world", len(good))
    two_blocks = raw(1, b"ab") + raw(1, b"cd") + b"\x00garbage"
    assert walk(two_blocks)[:3] == (0, 4, 2) and walk(two_blocks)[3] == len(two_blocks) - 7
    assert walk(b"\x00") == (0, 0, 0, 1) and H.oracle_lzma2_decompress(b"\x00", 0, 0) == (b"", 1)
    lz = lambda ctl: bytes([ctl, 0, 0, 0, 4]) + (b"\x5d" if ctl >= 0xC0 else b"") + bytes(5) + b"\x00"    # header of a 1-byte LZMA chunk, dummy payload
    bad = [
        b"",                                   # no end marker
        raw(2, b"x") + b"\x00",                # first chunk without a dictionary reset
        raw(1, b"x"),                          # truncated: end marker missing
        raw(1, b"x")[:-1],                     # truncated payload
        b"\x03\x00\x00x\x00",                  # control bytes 3..0x7F do not exist
        lz(0x80), lz(0xA0), lz(0xC0),          # LZMA chunk before any dictionary reset
        raw(1, b"x") + lz(0x80), raw(1, b"x") + lz(0xA0),      # after an uncompressed reset the next LZMA chunk needs new properties (>= 0xC0)
        bytes([0xE0, 0, 0, 0, 4, 225]) + bytes(5) + b"\x00",   # property byte out of range
        bytes([0xE0, 0, 0, 0, 4, 4 * 9 + 8 + 0]) + bytes(5) + b"\x00",   # lc 8 + lp 4 > 4
    ]
    for b in bad:
        assert walk(b)[0] == -5, b
        with pytest.raises(ValueError):
            H.oracle_lzma2_decompress(b, 64, 0)
