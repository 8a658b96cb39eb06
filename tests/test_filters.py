"""Delta and the stateless branch converters (ARM64, ARM, PPC, SPARC) -- csrc/b2z_filter.cu, SURVEY.md 8(f) item 3.
CPU: the oracle's statements (oracle/filter_oracle.c) against the REFERENCE's own converters (C/Bra.c z7_BranchConv_*_Enc/_Dec,
C/Delta.c, compiled into oracle/_ref/libref_xz.so) on instruction-dense data, word by word; decode(encode(x)) == x; the kernel
sources through the host emulation (tests/cuemu).  The GPU test of the C ABI is tests/test_gpu_zzz_filters.py."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import helpers as H

HERE = os.path.dirname(os.path.abspath(__file__))
DELTA, ARM64, PPC, ARM, SPARC, X86, ARMT = 0x03, 0x0A, 0x03030205, 0x03030501, 0x03030805, 0x03030103, 0x03030701
REF_NAME = {ARM64: "ARM64", ARM: "ARM", PPC: "PPC", SPARC: "SPARC", ARMT: "ARMT"}


def oracle_filter(method, enc, data, prop):
    O = H.oracle()
    O.b2zo_filter.argtypes = [ctypes.c_uint32, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32]
    buf = np.frombuffer(bytearray(data), dtype=np.uint8)
    assert O.b2zo_filter(method, enc, buf.ctypes.data if len(data) else None, len(data), prop) == 0
    return buf.tobytes()


def ref_filter(method, enc, data, prop):
    """digest of what the reference's converter makes of `data` (recorded where the reference is absent)"""
    return H.reference_answer("filter", (method, enc, data, prop), lambda: H.digest(_ref_filter(method, enc, data, prop)), H.ref_xz_available())


def _ref_filter(method, enc, data, prop):
    R = ctypes.CDLL(os.path.join(H.ROOT, "oracle", "_ref", "libref_xz.so"))
    buf = np.frombuffer(bytearray(data), dtype=np.uint8)
    if method == DELTA:
        state = ctypes.create_string_buffer(256)
        R.Delta_Init(state)
        f = R.Delta_Encode if enc else R.Delta_Decode
        f.argtypes = [ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p, ctypes.c_size_t]
        f(state, prop, buf.ctypes.data, len(data))
    elif method == X86:
        f = R.z7_BranchConvSt_X86_Enc if enc else R.z7_BranchConvSt_X86_Dec
        f.restype = ctypes.c_void_p; f.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.POINTER(ctypes.c_uint32)]
        state = ctypes.c_uint32(0)
        f(buf.ctypes.data, len(data), prop, ctypes.byref(state))
    else:
        f = getattr(R, f"z7_BranchConv_{REF_NAME[method]}_{'Enc' if enc else 'Dec'}")
        f.restype = ctypes.c_void_p; f.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32]
        end = f(buf.ctypes.data, len(data), prop)
        if method != ARMT:
            assert end - buf.ctypes.data == (len(data) & ~3)        # processes whole instructions, leaves the tail
    return buf.tobytes()


def instruction_soup(method, n_words, seed):
    """words that hit the converters' patterns often, with immediates at and around every range boundary"""
    rng = random.Random(seed); out = bytearray()
    for _ in range(n_words):
        r = rng.random(); w = rng.getrandbits(32)
        if method == ARM64:
            if r < 0.3: w = 0x94000000 | rng.getrandbits(26)
            elif r < 0.7:
                imm = rng.choice([0, 1, -1, (1 << 17) - 1, 1 << 17, -(1 << 17), -(1 << 17) - 1, (1 << 20) - 1, -(1 << 20), rng.getrandbits(21) - (1 << 20), rng.getrandbits(18) - (1 << 17)]) & 0x1FFFFF
                w = 0x90000000 | ((imm & 3) << 29) | ((imm >> 2) << 5) | rng.getrandbits(5)
            le = True
        elif method == ARM:
            if r < 0.5: w = 0xEB000000 | rng.getrandbits(24)
            le = True
        elif method == PPC:
            if r < 0.5: w = 0x48000001 | (rng.getrandbits(24) << 2)
            elif r < 0.6: w = 0x48000000 | rng.getrandbits(26)
            le = False
        elif method == ARMT:                                        # halfword pairs: BL pairs, lone first / second halves, chains F8xx F0xx F8xx
            h0 = rng.getrandbits(16); h1 = rng.getrandbits(16)
            if r < 0.4: h0 = 0xF000 | rng.getrandbits(11); h1 = 0xF800 | rng.getrandbits(11)
            elif r < 0.6: h0 = 0xF800 | rng.getrandbits(11); h1 = 0xF000 | rng.getrandbits(11)
            elif r < 0.7: h0 = 0xF000 | rng.getrandbits(11)
            out += h0.to_bytes(2, "little") + h1.to_bytes(2, "little")
            continue
        else:
            if r < 0.3: w = 0x40000000 | rng.getrandbits(22)
            elif r < 0.6: w = 0x7FC00000 | rng.getrandbits(22)
            elif r < 0.7: w = 0x40000000 | rng.getrandbits(30)
            le = False
        out += w.to_bytes(4, "little" if le else "big")
    return bytes(out)


@pytest.mark.parametrize("method", [ARM64, ARM, PPC, SPARC, ARMT])
def test_branch_converters_equal_the_reference(method):
    for seed, prop in ((1, 0), (2, 0x1000), (3, 0xFFFFF000), (4, 0x12345678), (5, 0x7FFFFFFC), (6, 0xFFFFFFFC)):
        data = instruction_soup(method, 60_000, seed) + b"\x94\x00\x00"[: seed % 4]      # ragged tail stays untouched
        enc = oracle_filter(method, 1, data, prop)
        assert enc != data and oracle_filter(method, 0, enc, prop) == data       # start offsets are multiples of 4: the coders reject
                                                                                   # others (BranchMisc.cpp:57,99), as b200z_filter_device does
        assert H.digest(enc) == ref_filter(method, 1, data, prop), (hex(method), hex(prop))
        assert H.digest(oracle_filter(method, 0, data, prop)) == ref_filter(method, 0, data, prop)     # decoding arbitrary words agrees too


def x86_soup(n, density, seed):
    """bytes dense in E8 / E9 opcodes and 00 / FF operand tops: long chains of overlapping candidates"""
    rng = random.Random(seed)
    return bytes(rng.choice([0xE8, 0xE9]) if rng.random() < density else (rng.choice([0, 0xFF]) if rng.random() < 0.4 else rng.randrange(256)) for _ in range(n))


def call_heavy_code(n, seed):
    """x86-like bytes where BCJ pays: a CALL rel32 every 16 bytes to one of 64 absolute targets -- the relative operands all
    differ, the absolute ones repeat"""
    rng = random.Random(seed); targets = [rng.randrange(0, n) for _ in range(64)]
    out = bytearray(rng.choice(b"\x8b\x45\x89\x55\x48\x83\xc4\x10") for _ in range(n))
    for pos in range(0, n - 5, 16):
        rel = (rng.choice(targets) - (pos + 5)) & 0xFFFFFFFF
        out[pos] = 0xE8; out[pos + 1:pos + 5] = rel.to_bytes(4, "little")
    return bytes(out)


def test_x86_bcj_pays_on_call_heavy_code(pkg):
    data = call_heavy_code(1 << 20, 3)
    filtered = oracle_filter(X86, 1, data, 0)
    assert oracle_filter(X86, 0, filtered, 0) == data
    plain = len(H.oracle_lzma2_compress(data)[1]); bcj = len(H.oracle_lzma2_compress(filtered)[1])
    assert bcj < 0.8 * plain, (plain, bcj)


def test_x86_bcj_equals_the_reference():
    rng = random.Random(2); cases = []
    for it in range(1200):
        n = rng.choice([0, 1, 4, 5, 6, 9, 17, 100, 1000, 5000]); pc = rng.choice([0, 0x1000, 0xFFFFFF00, rng.getrandbits(32)])
        data = x86_soup(n, rng.choice([0.02, 0.2, 0.5]), it)
        enc = oracle_filter(X86, 1, data, pc)
        assert oracle_filter(X86, 0, enc, pc) == data
        cases += [(X86, e, data, pc) for e in (1, 0)]
    # one recorded answer for all 2 400 conversions: the digest of their digests
    want = H.reference_answer("x86_filters", [x for c in cases for x in c], lambda: H.digest("".join(H.digest(_ref_filter(*c)) for c in cases).encode()), H.ref_xz_available())
    assert H.digest("".join(H.digest(oracle_filter(*c)) for c in cases).encode()) == want


def test_liblzma_filters_agree(pkg):
    """an implementation that shares no code with the reference: what liblzma's filters write (read back through a raw LZMA2-only
    decode) is undone by the oracle's statements -- the xz reader relies on exactly this"""
    import lzma
    lz2 = {"id": lzma.FILTER_LZMA2, "preset": 0}
    cases = [(X86, {"id": lzma.FILTER_X86}, x86_soup(200_003, 0.1, 3), 0), (X86, {"id": lzma.FILTER_X86, "start_offset": 0x1000}, x86_soup(50_000, 0.4, 4), 0x1000),
             (ARM, {"id": lzma.FILTER_ARM}, instruction_soup(ARM, 30_000, 5), 0), (PPC, {"id": lzma.FILTER_POWERPC}, instruction_soup(PPC, 30_000, 6), 0),
             (SPARC, {"id": lzma.FILTER_SPARC}, instruction_soup(SPARC, 30_000, 7), 0), (ARMT, {"id": lzma.FILTER_ARMTHUMB}, instruction_soup(ARMT, 30_000, 8), 0), (DELTA, {"id": lzma.FILTER_DELTA, "dist": 7}, pkg.corpus.entropy_class(2, 100_000).tobytes(), 7)]
    for method, f, data, prop in cases:
        filtered = lzma.decompress(lzma.compress(data, format=lzma.FORMAT_RAW, filters=[f, lz2]), format=lzma.FORMAT_RAW, filters=[lz2])
        assert filtered == oracle_filter(method, 1, data, prop), hex(method)
        assert oracle_filter(method, 0, filtered, prop) == data


def test_delta_equals_the_reference(pkg):
    data = pkg.corpus.entropy_class(2, 100_001).tobytes() + bytes(range(256)) * 40
    for dist in (1, 2, 3, 4, 7, 16, 255, 256):
        for n in (0, 1, dist - 1 if dist > 1 else 1, dist, dist + 1, 1000, len(data)):
            d = data[:n]
            enc = oracle_filter(DELTA, 1, d, dist)
            assert oracle_filter(DELTA, 0, enc, dist) == d
            assert H.digest(enc) == ref_filter(DELTA, 1, d, dist), (dist, n)
            assert H.digest(oracle_filter(DELTA, 0, d, dist)) == ref_filter(DELTA, 0, d, dist)


def test_emulated_kernels_equal_the_oracle(pkg):
    E = H.cuemu_library()
    E.emu_filter.restype = None; E.emu_filter.argtypes = [ctypes.c_uint32, ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32]

    def emu(method, enc, data, prop, unit_log=0):
        buf = np.frombuffer(bytearray(data) + bytearray(8), dtype=np.uint8)
        E.emu_filter(method, enc, buf.ctypes.data, len(data), prop, unit_log)
        return buf[:len(data)].tobytes()
    # per-unit encoding (the xz writer filters every Block on its own): equals the oracle applied unit by unit
    for method, data, prop in ((X86, x86_soup(3 * 4096 + 1001, 0.3, 8), 0), (ARMT, instruction_soup(ARMT, 3 * 1024 + 100, 8), 0x100), (ARM64, instruction_soup(ARM64, 3 * 1024 + 100, 8), 0x1000),
                               (DELTA, bytes((i * 7) & 0xFF for i in range(3 * 4096 + 5)), 3)):
        want = b"".join(oracle_filter(method, 1, data[i:i + 4096], prop) for i in range(0, len(data), 4096))
        assert emu(method, 1, data, prop, 12) == want, hex(method)
    for method in (ARM64, ARM, PPC, SPARC, ARMT):
        data = instruction_soup(method, 20_000, 9) + b"\x01\x02"
        for enc in (1, 0):
            assert emu(method, enc, data, 0x00ABC000) == oracle_filter(method, enc, data, 0x00ABC000), (hex(method), enc)
            assert emu(method, enc, data, 0xFFFFF000) == oracle_filter(method, enc, data, 0xFFFFF000), (hex(method), enc, "addresses that wrap")
    for seed, dens in ((1, 0.02), (2, 0.2), (3, 0.5), (4, 0.9)):       # x86: sparse opcodes ... one endless cluster
        for n in (0, 4, 5, 31, 32, 33, 37, 100, 4096, 70_001):
            data = x86_soup(n, dens, seed * 100 + n % 7)
            for enc in (1, 0):
                assert emu(X86, enc, data, 0x00400000) == oracle_filter(X86, enc, data, 0x00400000), (dens, n, enc)
    data = pkg.corpus.entropy_class(2, 300_001).tobytes()
    for dist in (1, 3, 4, 255, 256):
        for n in (1, dist, 65536, 65537, len(data)):                 # around the 64 KiB tiles of the decoder
            d = data[:n]
            assert emu(DELTA, 1, d, dist) == oracle_filter(DELTA, 1, d, dist), (dist, n)
            assert emu(DELTA, 0, d, dist) == oracle_filter(DELTA, 0, d, dist), (dist, n)
