"""The drop-in boundary: the C-ABI library exports every symbol include/b200z.h declares, the
7-Zip codec module exports the loader's entry points with the reference's method properties
(CPU, no compute), and -- on a GPU -- ICompressCoder::Code() round-trips through the module and
the reference decoder accepts what it wrote."""
import ctypes
import os
import re
import subprocess

import pytest

import helpers

ROOT = helpers.ROOT
PKG = os.path.join(ROOT, "7-zip-zstd_b200")


def test_c_abi_exports_match_header():
    hdr = open(os.path.join(ROOT, "include", "b200z.h")).read()
    declared = set(re.findall(r"\b(b200z_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    lib = ctypes.CDLL(os.path.join(PKG, "libb200z.so"))          # loading needs libcudart only, no GPU
    missing = [n for n in sorted(declared) if not hasattr(lib, n)]
    assert not missing, missing


def test_no_device_fails_loudly(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.B200zError):
        pkg.Codec(0)                                                # no CPU fallback


def test_codec_module_exports():
    out = subprocess.run([os.path.join(PKG, "build", "coder_roundtrip"), os.path.join(PKG, "libb200z_7z.so"), "--exports", "x"],
                         capture_output=True, text=True, timeout=60)
    assert out.returncode == 0 and "exports ok" in out.stdout, out.stderr


def test_frame_info_host_only():
    lib = ctypes.CDLL(os.path.join(PKG, "libb200z.so"))
    lib.b200z_zstd_frame_info.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32)]
    comp = helpers.oracle_compress(b"abc" * 100000, frameLog=17, windowLog=17, flags=1)
    cs, nf = ctypes.c_uint64(), ctypes.c_uint32()
    buf = ctypes.create_string_buffer(comp, len(comp))
    assert lib.b200z_zstd_frame_info(buf, len(comp), ctypes.byref(cs), ctypes.byref(nf)) == 0
    assert cs.value == 300000 and nf.value == 3
    assert lib.b200z_zstd_frame_info(buf, len(comp) - 5, ctypes.byref(cs), ctypes.byref(nf)) == -5


@pytest.mark.gpu
def test_icompresscoder_roundtrip(pkg, tmp_path):
    data = pkg.corpus.g2(5 * (1 << 20) + 999).tobytes() + bytes(300000)
    src = tmp_path / "in.bin"; packed = tmp_path / "packed.zst"
    src.write_bytes(data)
    out = subprocess.run([os.path.join(PKG, "build", "coder_roundtrip"), os.path.join(PKG, "libb200z_7z.so"), str(src), str(packed), "3"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "roundtrip ok" in out.stdout, out.stderr + out.stdout
    comp = packed.read_bytes()
    assert comp[:4] == b"\x50\x2a\x4d\x18"                            # mcmilk MT size hint in front of the first frame
    assert helpers.oracle_decompress(comp, len(data)) == data
    assert helpers.ref_zstd_result(comp, len(data)) == helpers.digest(data)


def codec_module_lzma2_roundtrip(pkg, tmp_path, method, level, price_parse):
    """Method 21 through the codec module (CreateEncoder/CreateDecoder by index, as LoadCodecs.cpp does); the packed
    stream must also be accepted by the reference decoder and liblzma.  The level picks the parse as the reference's
    normalisation does (LzmaEnc.c:97 algo = level < 5 ? 0 : 1; fast-lzma2's table: fast below level 3)."""
    import lzma
    data = pkg.corpus.g2(3 * (1 << 20) + 777).tobytes() + bytes(200000) + pkg.corpus.entropy_class(1, 150000).tobytes()
    src = tmp_path / "in.bin"; packed = tmp_path / "packed.lzma2"
    src.write_bytes(data)
    out = subprocess.run([os.path.join(PKG, "build", "coder_roundtrip"), os.path.join(PKG, "libb200z_7z.so"), str(src), str(packed), str(level), method],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "roundtrip ok" in out.stdout, out.stderr + out.stdout
    comp = packed.read_bytes()
    assert lzma.LZMADecompressor(format=lzma.FORMAT_RAW, filters=[{"id": lzma.FILTER_LZMA2, "dict_size": 1 << 20}]).decompress(comp) == data
    assert helpers.ref_lzma2_result(comp, len(data), 16) == (helpers.digest(data), len(comp))
    assert comp == helpers.oracle_lzma2_compress(data, flags=1 | (2 << 8) | (0x10 if price_parse else 0))[1]


@pytest.mark.gpu
@pytest.mark.parametrize("method,level", [("lzma2", 4), ("flzma2", 2)])
def test_icompresscoder_roundtrip_lzma2(pkg, tmp_path, method, level):
    """levels below the reference's switch to its optimal parsers: the greedy parse (the price-based parse at levels >= 5 / 3 is
    covered by tests/test_gpu_zz_lzma2_parse.py)"""
    codec_module_lzma2_roundtrip(pkg, tmp_path, method, level, False)


def test_binding_parameter_ids_match_header(pkg):
    """The ctypes binding names parameters by number: they must be the header's B200Z_P_* values."""
    hdr = open(os.path.join(ROOT, "include", "b200z.h")).read()
    ids = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+B200Z_P_([A-Z0-9_]+)\s+(\d+)", hdr)}
    names = dict(level="LEVEL", frame_log="FRAMELOG", hash_log_l="HASHLOG_L", hash_log_s="HASHLOG_S", window_log="WINDOWLOG", flags="FLAGS",
                 batch_log="BATCH_LOG", host_batch_log="HOST_BATCH_LOG", chunk_log="CHUNKLOG", lzma2_model="LZMA2_MODEL", lzma2_slice_log="LZMA2_SLICELOG",
                 lzma2_parse="LZMA2_PARSE", zstd_parse="ZSTD_PARSE", long="LONG", region_log="REGIONLOG", dec_jump="DEC_JUMP", dec_jump_seg_log="DEC_JUMP_SEGLOG")
    assert set(names) == set(pkg.Codec._PARAMS)
    for k, h in names.items():
        assert pkg.Codec._PARAMS[k] == ids[h], k
    assert len(set(ids.values())) == len(ids)


def _abi_facts(tmp_path, *flags):
    exe = str(tmp_path / ("abi_" + str(len(flags))))
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wno-invalid-offsetof", *flags, os.path.join(ROOT, "tests", "cpp", "abi_facts.cpp"), "-o", exe])
    return subprocess.check_output([exe]).decode()


def test_abi_declaration_equals_the_reference_headers(tmp_path):
    """codec/b2z_7zip_abi.h re-declares the codec-plugin ABI so that the module builds without the 7-Zip tree; this compiles the same
    fact printer (struct layout, HRESULTs, interface IDs, every NCoderPropID / NMethodPropID value, the ZSTD level bytes, the vtable
    slot of every interface method) against it AND against the reference's own MyWindows.h / MyCom.h / ICoder.h / IStream.h.
    Where /root/reference is absent the committed copy of the reference's output (tests/golden/abi_facts_reference.txt) stands in."""
    ours = _abi_facts(tmp_path)
    golden = os.path.join(ROOT, "tests", "golden", "abi_facts_reference.txt")
    if os.path.isdir("/root/reference/CPP/7zip"):
        ref = _abi_facts(tmp_path, "-DB2Z_REFERENCE_HEADERS", "-I/root/reference/CPP")
        assert ref == open(golden).read(), "tests/golden/abi_facts_reference.txt is stale: regenerate it with abi_facts.cpp -DB2Z_REFERENCE_HEADERS"
    else:
        ref = open(golden).read()
    assert ours == ref
    assert "ultimate 255 fast_inc 32" in ours and "slot ICompressCoder::Code 3" in ours
