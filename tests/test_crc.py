"""CRC32 (7-Zip's file / folder digest, C/7zCrc.c CrcCalc) and CRC-64/XZ (xz block check, C/XzCrc64.c) -- csrc/b2z_crc.cu.
CPU: the oracle statements against the check values, zlib and the reference's own functions; the library's host-side combine
arithmetic; the kernel source through the host emulation (tests/cuemu).  The GPU test of the C ABI is tests/test_gpu_zzz_crc.py."""
import ctypes
import os
import random
import subprocess
import zlib

import numpy as np
import pytest

import helpers as H

HERE = os.path.dirname(os.path.abspath(__file__))


def _oracle():
    O = H.oracle()
    O.b2zo_crc32.restype = ctypes.c_uint32; O.b2zo_crc32.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
    O.b2zo_crc64.restype = ctypes.c_uint64; O.b2zo_crc64.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
    return O


def _ref_xz():
    L = ctypes.CDLL(os.path.join(H.ROOT, "oracle", "_ref", "libref_xz.so"))
    L.CrcGenerateTable(); L.Crc64GenerateTable()
    L.CrcCalc.restype = ctypes.c_uint32; L.CrcCalc.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
    L.Crc64Update.restype = ctypes.c_uint64; L.Crc64Update.argtypes = [ctypes.c_uint64, ctypes.c_char_p, ctypes.c_size_t]
    return L


def test_oracle_pinned_to_check_values_zlib_and_the_reference(pkg):
    O = _oracle()
    assert O.b2zo_crc32(b"123456789", 9) == 0xCBF43926 and O.b2zo_crc64(b"123456789", 9) == 0x995DC9BBDF1939FA
    assert O.b2zo_crc32(b"", 0) == 0 and O.b2zo_crc64(b"", 0) == 0
    for name, data in H.sample_inputs(pkg).items():
        assert O.b2zo_crc32(data, len(data)) == zlib.crc32(data), name

        def ask():
            L = _ref_xz()
            return L.CrcCalc(data, len(data)), L.Crc64Update(0xFFFFFFFFFFFFFFFF, data, len(data)) ^ 0xFFFFFFFFFFFFFFFF
        assert H.reference_answer("crc32_crc64", (data,), ask, H.ref_xz_available()) == (O.b2zo_crc32(data, len(data)), O.b2zo_crc64(data, len(data))), name


def test_library_combine_arithmetic(pkg):
    """crc(A || B) from crc(A), crc(B), |B| -- the fold the whole-buffer digests use (host code of libb200z.so, no device)."""
    O = _oracle(); L = pkg.load_library()
    L.b200z_crc32_combine.restype = ctypes.c_uint32; L.b200z_crc32_combine.argtypes = [ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint64]
    L.b200z_crc64_combine.restype = ctypes.c_uint64; L.b200z_crc64_combine.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64]
    rng = random.Random(7)
    data = pkg.corpus.g2(300_000).tobytes() + bytes(1000) + pkg.corpus.entropy_class(1, 100_000).tobytes()
    for _ in range(40):
        a = rng.randrange(0, len(data)); b = rng.randrange(a, len(data) + 1)
        A, B = data[:a], data[a:b]
        assert L.b200z_crc32_combine(zlib.crc32(A), zlib.crc32(B), len(B)) == zlib.crc32(A + B)
        assert L.b200z_crc64_combine(O.b2zo_crc64(A, len(A)), O.b2zo_crc64(B, len(B)), len(B)) == O.b2zo_crc64(A + B, len(A) + len(B))


def test_emulated_kernel_equals_the_oracle(pkg):
    E = H.cuemu_library()
    vp, u32, u64 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64
    E.emu_crc_pieces.restype = u64; E.emu_crc_pieces.argtypes = [vp, u64, u32, vp, vp, u32, u32, vp]
    O = _oracle()
    data = pkg.corpus.g2(200_000).tobytes() + pkg.corpus.entropy_class(1, 70_001).tobytes()
    n = len(data); src = np.frombuffer(data + bytes(64), dtype=np.uint8)
    for plog in (12, 16):                                          # fixed pieces; the last one is ragged
        np_ = (n + (1 << plog) - 1) >> plog
        for width, dt, f in ((32, np.uint32, O.b2zo_crc32), (64, np.uint64, O.b2zo_crc64)):
            out = np.zeros(np_, dtype=dt)
            E.emu_crc_pieces(src.ctypes.data, n, plog, None, None, np_, width, out.ctypes.data)
            for i in range(np_):
                piece = data[i << plog:(i + 1) << plog]
                assert int(out[i]) == f(piece, len(piece)), (plog, width, i)
    rng = random.Random(3)                                         # caller-given ranges at any alignment, empty ones included
    offs = np.array([rng.randrange(0, n - 5000) for _ in range(200)], dtype=np.uint64)
    lens = np.array([rng.choice([0, 1, 7, 8, 9, 63, 64, 1000, 4999]) for _ in range(200)], dtype=np.uint64)
    for width, dt, f in ((32, np.uint32, O.b2zo_crc32), (64, np.uint64, O.b2zo_crc64)):
        out = np.zeros(200, dtype=dt)
        E.emu_crc_pieces(src.ctypes.data, n, 0, offs.ctypes.data, lens.ctypes.data, 200, width, out.ctypes.data)
        for i in range(200):
            piece = data[int(offs[i]):int(offs[i]) + int(lens[i])]
            assert int(out[i]) == f(piece, len(piece)), (width, i)


def test_emulated_sha256_kernel_equals_hashlib(pkg):
    """the third xz check type (C/Xz.h:35 XZ_CHECK_SHA256): sha256_pieces_kernel, one thread per range, every padding case"""
    import hashlib
    E = H.cuemu_library()
    E.emu_sha256_pieces.restype = None; E.emu_sha256_pieces.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_uint32, ctypes.c_void_p]
    rng = random.Random(1); data = pkg.corpus.entropy_class(1, 30_000).tobytes()
    lens = [0, 1, 54, 55, 56, 57, 63, 64, 65, 119, 120, 127, 128, 1000, 4097, 20_000]; offs = [rng.randrange(0, 10_000) for _ in lens]
    o = np.array(offs, dtype=np.uint64); ln = np.array(lens, dtype=np.uint64); out = np.zeros(len(lens) * 8, dtype=np.uint32)
    src = np.frombuffer(data, dtype=np.uint8)
    E.emu_sha256_pieces(src.ctypes.data, o.ctypes.data, ln.ctypes.data, len(lens), out.ctypes.data)
    for i in range(len(lens)):
        assert b"".join(int(w).to_bytes(4, "big") for w in out[i * 8:i * 8 + 8]) == hashlib.sha256(data[offs[i]:offs[i] + lens[i]]).digest(), lens[i]
