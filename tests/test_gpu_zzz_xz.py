"""GPU: the .xz container around the GPU LZMA2 coder (csrc/xz_api.cu) through the C ABI: files we write are decoded and verified
by liblzma and the reference's unpacker; files liblzma writes (and our own) are decoded by the GPU with their Block checks
verified; damage is reported.  Sorts last: first hardware run of this path (written after the round's GPU budget was spent; the
container logic and the CRC kernel are checked on the CPU in tests/test_xz_container.py and tests/test_crc.py)."""
import lzma

import numpy as np
import pytest

import helpers as H
from test_xz_container import ref_unpack

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def inputs(pkg):
    return H.sample_inputs(pkg, big=False)


def test_files_we_write_decode_everywhere(pkg, codec, inputs):
    for name, data in inputs.items():
        for check in (0, 1, 4):
            xz = codec.xz_compress(data, check)
            assert lzma.decompress(xz, format=lzma.FORMAT_XZ) == data, (name, check)
            assert codec.xz_decompress(xz) == data, (name, check)
        r = ref_unpack(codec.xz_compress(data, 4), len(data))
        assert r[0] == 0 and r[1] == H.digest(data) and r[3] != 0, name
    c = pkg.Codec(0, frame_log=18, window_log=18, lzma2_parse=1)     # price-based parse, 256 KiB Blocks
    data = inputs["mixed"] + inputs["g2_1m"]
    xz = c.xz_compress(data)
    assert lzma.decompress(xz, format=lzma.FORMAT_XZ) == data and c.xz_decompress(xz) == data
    c.close()


def test_writer_with_a_gpu_filter_per_block(pkg, codec):
    from test_filters import x86_soup, instruction_soup
    exe = x86_soup(3 * (1 << 20) + 12_345, 0.04, 11)
    for fid, fprop, data in ((0x03030103, 0, exe), (0x03, 4, bytes((i * 5) & 0xFF for i in range((2 << 20) + 77))), (0x03030501, 0, instruction_soup(0x03030501, 600_000, 12))):
        xz = codec.xz_compress(data, 4, fid, fprop)
        assert lzma.decompress(xz, format=lzma.FORMAT_XZ) == data, hex(fid)       # liblzma undoes the filter and verifies the CRC64 of the original
        assert codec.xz_decompress(xz) == data, hex(fid)
    from test_filters import call_heavy_code
    code = call_heavy_code(2 << 20, 3)
    plain = codec.xz_compress(code, 4); bcj = codec.xz_compress(code, 4, 0x03030103, 0)
    assert len(bcj) < 0.8 * len(plain) and lzma.decompress(bcj, format=lzma.FORMAT_XZ) == code      # absolute call targets repeat; relative ones do not


def test_foreign_files_and_damage(pkg, codec, inputs):
    data = inputs["g2_1m"]
    for check in (lzma.CHECK_NONE, lzma.CHECK_CRC32, lzma.CHECK_CRC64, lzma.CHECK_SHA256):
        assert codec.xz_decompress(lzma.compress(data, format=lzma.FORMAT_XZ, check=check, preset=1)) == data
    # filter chains in front of LZMA2 are undone on the GPU (x86-dense and delta-friendly payloads so that the filters do something)
    from test_filters import x86_soup, instruction_soup
    lz2 = {"id": lzma.FILTER_LZMA2, "preset": 1}
    exe = x86_soup(500_003, 0.05, 5); ramp = bytes((i * 3) & 0xFF for i in range(400_001))
    for payload, filt in ((exe, [{"id": lzma.FILTER_X86}]), (exe, [{"id": lzma.FILTER_X86, "start_offset": 0x1000}]), (ramp, [{"id": lzma.FILTER_DELTA, "dist": 3}]),
                          (exe, [{"id": lzma.FILTER_ARM}]), (instruction_soup(0x03030701, 100_000, 3), [{"id": lzma.FILTER_ARMTHUMB}]), (exe, [{"id": lzma.FILTER_POWERPC}]), (exe, [{"id": lzma.FILTER_SPARC}]),
                          (ramp + exe, [{"id": lzma.FILTER_DELTA, "dist": 1}, {"id": lzma.FILTER_X86}])):
        xzf = lzma.compress(payload, format=lzma.FORMAT_XZ, filters=filt + [lz2])
        assert codec.xz_decompress(xzf) == payload, filt
    two = lzma.compress(exe[:100_001], format=lzma.FORMAT_XZ, filters=[{"id": lzma.FILTER_X86}, lz2]) + lzma.compress(exe[100_001:], format=lzma.FORMAT_XZ, filters=[{"id": lzma.FILTER_ARM}, lz2])
    assert codec.xz_decompress(two) == exe                            # second Stream's Block starts at an odd offset: staged for alignment
    with pytest.raises(pkg.B200zError) as e:
        codec.xz_decompress(lzma.compress(exe[:1000], format=lzma.FORMAT_XZ, filters=[{"id": lzma.FILTER_IA64}, lz2]))
    assert e.value.code == -6
    a = lzma.compress(data[:300_000], format=lzma.FORMAT_XZ); b = lzma.compress(data[300_000:], format=lzma.FORMAT_XZ, check=lzma.CHECK_CRC32, preset=0)
    assert codec.xz_decompress(a + bytes(8) + b) == data              # concatenated Streams
    sha = bytearray(lzma.compress(data, format=lzma.FORMAT_XZ, check=lzma.CHECK_SHA256, preset=1))
    sha[-40] ^= 1                                                     # inside the 32 check bytes: the GPU's SHA-256 disagrees
    with pytest.raises(pkg.B200zError) as e:
        codec.xz_decompress(bytes(sha))
    assert e.value.code == -8
    xz = bytearray(codec.xz_compress(data, 4))
    xz[len(xz) // 2] ^= 0x10                                          # inside a Block's payload: the range decoder or the check notices
    with pytest.raises(pkg.B200zError) as e:
        codec.xz_decompress(bytes(xz))
    assert e.value.code in (-5, -8)
    with pytest.raises(pkg.B200zError):
        codec.xz_decompress(bytes(xz[:-5]))


def test_large_roundtrip_property(pkg, codec):
    data = pkg.corpus.g2(48 << 20, seed=80)
    xz = codec.xz_compress(data)
    out = codec.xz_decompress(xz)
    assert np.array_equal(np.frombuffer(out, dtype=np.uint8), data)
