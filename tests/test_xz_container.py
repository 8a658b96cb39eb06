"""CPU: the .xz container logic of csrc/xz_api.cu (b200z_xz_wrap / b200z_xz_parse: host code of libb200z.so, no device needed).
Writer: oracle LZMA2 streams (both parses) + per-frame CRC32 / CRC64 from the oracle -> .xz that liblzma (Python's lzma) and the
reference's own unpacker (C/XzDec.c via oracle/_ref/libref_xz.so) decode and VERIFY.  Reader: files written by liblzma (all check
types, concatenated streams, stream padding) and by our writer parse to the right Block table; damaged fields are rejected."""
import ctypes
import lzma
import os

import numpy as np
import pytest

import helpers as H

OPT = 0x10


class XzBlock(ctypes.Structure):
    _fields_ = [("packOff", ctypes.c_uint64), ("packSize", ctypes.c_uint64), ("unpackSize", ctypes.c_uint64), ("check", ctypes.c_uint64),
                ("dictProp", ctypes.c_uint32), ("checkType", ctypes.c_uint32), ("nFilters", ctypes.c_uint32),
                ("filterId", ctypes.c_uint32 * 3), ("filterProp", ctypes.c_uint32 * 3)]


def _lib(pkg):
    L = pkg.load_library()
    vp, sz, u32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32
    L.b200z_xz_wrap_bound.restype = sz; L.b200z_xz_wrap_bound.argtypes = [sz, u32]
    L.b200z_xz_wrap.argtypes = [vp, sz, u32, u32, vp, u32, u32, u32, vp, sz, ctypes.POINTER(sz)]
    L.b200z_xz_parse.argtypes = [vp, sz, ctypes.POINTER(XzBlock), u32, ctypes.POINTER(u32), ctypes.POINTER(ctypes.c_uint64)]
    return L


def _crc(kind, data):
    O = H.oracle()
    O.b2zo_crc32.restype = ctypes.c_uint32; O.b2zo_crc32.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
    O.b2zo_crc64.restype = ctypes.c_uint64; O.b2zo_crc64.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
    return O.b2zo_crc32(data, len(data)) if kind == 1 else (O.b2zo_crc64(data, len(data)) if kind == 4 else 0)


def _wrap(L, lz, prop, kind, data, fl, filter_id=0, filter_prop=0):
    F = 1 << fl
    checks = np.array([_crc(kind, data[i:i + F]) for i in range(0, len(data), F)] or [0], dtype=np.uint64)
    src = np.frombuffer(lz, dtype=np.uint8)
    cap = L.b200z_xz_wrap_bound(len(lz), len(checks)); out = np.zeros(cap, dtype=np.uint8); n = ctypes.c_size_t()
    rc = L.b200z_xz_wrap(src.ctypes.data, len(lz), prop, kind, checks.ctypes.data, len(checks), filter_id, filter_prop, out.ctypes.data, cap, ctypes.byref(n))
    assert rc == 0, rc
    return out[:n.value].tobytes()


def _parse(L, xz, cap=4096):
    src = np.frombuffer(xz, dtype=np.uint8)
    blocks = (XzBlock * cap)(); nb = ctypes.c_uint32(); total = ctypes.c_uint64()
    rc = L.b200z_xz_parse(src.ctypes.data, len(xz), blocks, cap, ctypes.byref(nb), ctypes.byref(total))
    return rc, [blocks[i] for i in range(min(nb.value, cap))], total.value


def ref_unpack(xz, n):
    """(status, digest of the output, bytes consumed, stream finished) of the reference's unpacker (recorded where it is absent)"""
    def ask():
        rc, out, used, fin = _ref_unpack(xz, n)
        return rc, H.digest(out), used, fin
    return H.reference_answer("xz_unpack", (xz, n), ask, H.ref_xz_available())


def _ref_unpack(xz, n):
    """the reference's unpacker (C/XzDec.c XzUnpacker_Code); verifies Block checks, Index and Footer"""
    R = ctypes.CDLL(os.path.join(H.ROOT, "oracle", "_ref", "libref_xz.so"))
    R.CrcGenerateTable(); R.Crc64GenerateTable()
    alloc = ctypes.c_void_p.in_dll(R, "g_Alloc")
    st = ctypes.create_string_buffer(1 << 16)                     # CXzUnpacker (opaque here; a few KB)
    R.XzUnpacker_Construct.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    R.XzUnpacker_Init.argtypes = [ctypes.c_void_p]; R.XzUnpacker_Free.argtypes = [ctypes.c_void_p]
    R.XzUnpacker_IsStreamWasFinished.argtypes = [ctypes.c_void_p]
    R.XzUnpacker_Code.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p, ctypes.POINTER(ctypes.c_size_t),
                                  ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
    R.XzUnpacker_Construct(st, ctypes.addressof(alloc)); R.XzUnpacker_Init(st)
    src = np.frombuffer(xz, dtype=np.uint8)
    out = bytearray(); ip = 0; chunk = np.zeros(1 << 20, dtype=np.uint8); status = ctypes.c_int(); rc = 0
    while True:                                                    # Interface-1 of C/Xz.h:296-308: partial output buffers
        dl = ctypes.c_size_t(chunk.size); sl = ctypes.c_size_t(len(xz) - ip)
        rc = R.XzUnpacker_Code(st, chunk.ctypes.data, ctypes.byref(dl), src.ctypes.data + ip, ctypes.byref(sl), 1, 0, ctypes.byref(status))
        out += chunk[:dl.value].tobytes(); ip += sl.value
        if rc != 0 or (dl.value == 0 and sl.value == 0):
            break
    fin = R.XzUnpacker_IsStreamWasFinished(st)
    R.XzUnpacker_Free(st)
    return rc, bytes(out), ip, fin


def test_writer_output_is_decoded_and_verified_by_liblzma_and_the_reference(pkg):
    L = _lib(pkg)
    data = pkg.corpus.g2(2 * (1 << 20) + 300_001).tobytes() + bytes(50_000) + pkg.corpus.entropy_class(1, 90_000).tobytes()
    for fl, flags in ((20, 1 | (2 << 8)), (18, 1 | (1 << 8) | OPT), (17, 1)):
        prop, lz = H.oracle_lzma2_compress(data, frameLog=fl, windowLog=fl, flags=flags)
        for kind in (0, 1, 4):
            xz = _wrap(L, lz, prop, kind, data, fl)
            assert lzma.decompress(xz, format=lzma.FORMAT_XZ) == data, (fl, kind)
            r = ref_unpack(xz, len(data))
            assert r[0] == 0 and r[1] == H.digest(data) and r[2] == len(xz) and r[3] != 0, (fl, kind, r[0])
            rc, blocks, total = _parse(L, xz)
            assert rc == 0 and total == len(data) and len(blocks) == (len(data) + (1 << fl) - 1) >> fl
            assert all(b.checkType == kind and b.dictProp == prop for b in blocks)
            assert [b.check for b in blocks] == [_crc(kind, data[i:i + (1 << fl)]) for i in range(0, len(data), 1 << fl)]
    # a wrong check value must be caught by the independent decoders
    prop, lz = H.oracle_lzma2_compress(data[:300_000])
    bad = bytearray(_wrap(L, lz, prop, 4, data[:300_000], 20)); rc, blocks, _ = _parse(L, bytes(bad))
    bad[blocks[0].packOff + ((blocks[0].packSize + 3) & ~3)] ^= 1
    with pytest.raises(lzma.LZMAError):
        lzma.decompress(bytes(bad), format=lzma.FORMAT_XZ)
    # empty input: a Stream with no Blocks
    prop, lz = H.oracle_lzma2_compress(b"")
    xz = _wrap(L, lz, prop, 4, b"", 20)
    assert lzma.decompress(xz, format=lzma.FORMAT_XZ) == b"" and _parse(L, xz)[:1] == (0,) and len(xz) == 32


def test_writer_with_a_filter_in_front_of_lzma2(pkg):
    """what b200z_xz_compress_host(filterId) assembles: every frame filtered on its own (oracle statements of the filters), the
    filtered bytes through the LZMA2 encoder statement, Blocks that declare the filter -- liblzma and the reference undo it and
    verify the checks of the ORIGINAL bytes"""
    from test_filters import oracle_filter, x86_soup, instruction_soup
    L = _lib(pkg); fl = 17; F = 1 << fl
    exe = x86_soup(3 * F + 12_345, 0.04, 11)
    for fid, fprop, data in ((0x03030103, 0, exe), (0x03030103, 0x1000, exe), (0x03, 4, bytes((i * 5) & 0xFF for i in range(2 * F + 77))),
                             (0x03030501, 0, instruction_soup(0x03030501, (2 * F + 64) // 4, 12)), (0x03030701, 0, instruction_soup(0x03030701, (2 * F + 64) // 4, 14)), (0x0A, 0x4000, instruction_soup(0x0A, (2 * F + 64) // 4, 13))):
        filtered = b"".join(oracle_filter(fid, 1, data[i:i + F], fprop) for i in range(0, len(data), F))
        prop, lz = H.oracle_lzma2_compress(filtered, frameLog=fl, windowLog=fl, flags=1)
        xz = _wrap(L, lz, prop, 4, data, fl, fid, fprop)
        if fid != 0x0A:                                             # this liblzma may predate the ARM64 filter
            assert lzma.decompress(xz, format=lzma.FORMAT_XZ) == data, hex(fid)
        r = ref_unpack(xz, len(data))
        assert r[0] == 0 and r[1] == H.digest(data) and r[3] != 0, hex(fid)
        rc, blocks, total = _parse(L, xz)
        assert rc == 0 and total == len(data) and all(b.nFilters == 1 and b.filterId[0] == fid and b.filterProp[0] == fprop for b in blocks)


def test_reader_parses_foreign_files_and_rejects_damage(pkg):
    L = _lib(pkg)
    data = pkg.corpus.g2(400_000).tobytes()
    for check, kind in ((lzma.CHECK_NONE, 0), (lzma.CHECK_CRC32, 1), (lzma.CHECK_CRC64, 4), (lzma.CHECK_SHA256, 10)):
        xz = lzma.compress(data, format=lzma.FORMAT_XZ, check=check, preset=1)
        rc, blocks, total = _parse(L, xz)
        assert rc == 0 and total == len(data) and len(blocks) == 1 and blocks[0].checkType == kind
        b = blocks[0]
        raw = xz[b.packOff:b.packOff + b.packSize]                # the Block's chunk stream decodes on its own
        assert H.oracle_lzma2_decompress(raw, len(data), b.dictProp) == (data, len(raw))
        if kind in (1, 4):
            assert b.check == _crc(kind, data)
    a = lzma.compress(data[:100_000], format=lzma.FORMAT_XZ); b = lzma.compress(data[100_000:], format=lzma.FORMAT_XZ, check=lzma.CHECK_CRC32)
    rc, blocks, total = _parse(L, a + bytes(8) + b + bytes(4))    # concatenated Streams with Stream Padding
    assert rc == 0 and len(blocks) == 2 and total == len(data) and (blocks[0].checkType, blocks[1].checkType) == (4, 1)
    xz = lzma.compress(data, format=lzma.FORMAT_XZ)
    assert _parse(L, xz[:-1])[0] == -5 and _parse(L, xz[:40])[0] == -5 and _parse(L, b"")[0] == -5
    for pos in (7, 9, 13, 20, len(xz) - 3, len(xz) - 9, len(xz) - 14):     # flags, header CRC, block header, footer fields, index
        bad = bytearray(xz); bad[pos] ^= 0x40
        assert _parse(L, bytes(bad))[0] in (-5, -6), pos
    assert _parse(L, a + bytes(3) + b)[0] == -5                   # Stream Padding must be a multiple of four bytes
    # filter chains: the ones the GPU can undo come back as 7-Zip method ids + property; the others are unsupported, not corrupt
    lz2 = {"id": lzma.FILTER_LZMA2, "preset": 1}
    for filt, want in (([{"id": lzma.FILTER_DELTA, "dist": 4}], [(0x03, 4)]), ([{"id": lzma.FILTER_X86}], [(0x03030103, 0)]),
                       ([{"id": lzma.FILTER_X86, "start_offset": 0x1000}], [(0x03030103, 0x1000)]), ([{"id": lzma.FILTER_ARM}], [(0x03030501, 0)]),
                       ([{"id": lzma.FILTER_POWERPC}], [(0x03030205, 0)]), ([{"id": lzma.FILTER_SPARC}], [(0x03030805, 0)]),
                       ([{"id": lzma.FILTER_ARMTHUMB}], [(0x03030701, 0)]),
                       ([{"id": lzma.FILTER_DELTA, "dist": 256}, {"id": lzma.FILTER_X86}], [(0x03, 256), (0x03030103, 0)])):
        rc, blocks, total = _parse(L, lzma.compress(data[:50_000], format=lzma.FORMAT_XZ, filters=filt + [lz2]))
        assert rc == 0 and total == 50_000 and blocks[0].nFilters == len(want), filt
        assert [(blocks[0].filterId[i], blocks[0].filterProp[i]) for i in range(len(want))] == want
    for filt in ([{"id": lzma.FILTER_IA64}],):
        assert _parse(L, lzma.compress(data[:50_000], format=lzma.FORMAT_XZ, filters=filt + [lz2]))[0] == -6


def test_reader_agrees_with_liblzma_on_damaged_container_fields(pkg):
    """differential check: a bit flip / overwritten byte in the Stream Header, a Block Header, the Index or the Footer is accepted by
    b200z_xz_parse exactly when liblzma still decodes the file to the original (20 000 mutants in a longer run: no disagreement)"""
    import random
    L = _lib(pkg)
    data = pkg.corpus.g2(300_000).tobytes()
    prop, lz = H.oracle_lzma2_compress(data, frameLog=17, windowLog=17, flags=1)
    seeds = [(lzma.compress(data[:50_000], format=lzma.FORMAT_XZ, preset=0), data[:50_000]), (_wrap(L, lz, prop, 4, data, 17), data), (_wrap(L, lz, prop, 1, data, 17), data)]
    rng = random.Random(9)
    for it in range(1500):
        xz, plain = rng.choice(seeds); s = bytearray(xz)
        rc0, blocks, _ = _parse(L, bytes(s))
        cb = {0: 0, 1: 4, 4: 8}[blocks[0].checkType]
        regions = [(0, 12)]; hs = 12
        for b in blocks:
            regions.append((hs, b.packOff)); hs = b.packOff + ((b.packSize + 3) & ~3) + cb
        regions.append((hs, len(s)))
        lo, hi = rng.choice(regions)
        pos = rng.randrange(lo, hi); s[pos] ^= 1 << rng.randrange(8)
        if rng.random() < 0.3:
            s[rng.randrange(lo, hi)] = rng.randrange(256)
        rc = _parse(L, bytes(s))[0]
        try:
            ok = lzma.decompress(bytes(s), format=lzma.FORMAT_XZ) == plain
        except lzma.LZMAError:
            ok = False
        assert (rc == 0) == ok, (it, pos, rc)


def test_reader_walks_every_block_payload(pkg):
    """a Block whose header declares both sizes is still walked chunk header by chunk header: an end marker before the declared
    Compressed Size, a chunk that runs past it, or chunk sizes that do not add up to the Uncompressed Size are rejected by the parser
    itself (as XzDec / liblzma reject them by decoding Block by Block), not left to whatever the spliced stream happens to decode to"""
    L = _lib(pkg)
    data = pkg.corpus.g2(600_000).tobytes()
    prop, lz = H.oracle_lzma2_compress(data, frameLog=18, windowLog=18, flags=1)        # 256 KiB Blocks: two chunks each
    xz = _wrap(L, lz, prop, 4, data, 18)
    rc, blocks, total = _parse(L, xz)
    assert rc == 0 and len(blocks) == 3 and total == len(data)
    b = blocks[1]
    def chunk_offsets(off, size):                                   # offsets of the chunk headers of one Block's payload
        out, ip = [], off
        while xz[ip] != 0:
            out.append(ip); c = xz[ip]
            ip += (3 + ((xz[ip + 1] << 8) | xz[ip + 2]) + 1) if c <= 2 else ((6 if c >= 0xC0 else 5) + ((xz[ip + 3] << 8) | xz[ip + 4]) + 1)
        assert ip == off + size - 1
        return out
    heads = chunk_offsets(b.packOff, b.packSize)
    assert len(heads) >= 2
    for mutate in (lambda s: s.__setitem__(heads[1], 0),                                   # end marker in the middle of the Block
                   lambda s: s.__setitem__(heads[-1] + 4, (s[heads[-1] + 4] + 1) & 255),    # last chunk one byte longer: runs over the end marker
                   lambda s: s.__setitem__(heads[-1] + 2, (s[heads[-1] + 2] + 1) & 255),    # chunk sizes no longer add up to the Uncompressed Size
                   lambda s: s.__setitem__(heads[0], 0x80)):                                # first chunk of a Block without a dictionary reset
        s = bytearray(xz); mutate(s)
        assert _parse(L, bytes(s))[0] == -5
        with pytest.raises(lzma.LZMAError):
            lzma.decompress(bytes(s), format=lzma.FORMAT_XZ)
