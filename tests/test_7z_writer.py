"""The .7z container writer of the many-files path (csrc/sevenz_api.cu, SURVEY.md 8(f) item 1 / BASELINE configs[4]).

CPU: b200z_7z_build_archive is host code -- fed with the ORACLE's frames (what the GPU emits, byte for byte) and zlib CRC32s it must
produce an archive the stock reference 7zz (oracle/_ref/7z/stock/7zz, built by oracle/build_ref_7z.sh) lists, tests and extracts:
names (non-ASCII included), sizes, CRCs, empty files, method string.  GPU (`-m gpu`): the one-call writer, same checks on 3 000 files."""
import ctypes
import os
import subprocess
import zlib

import numpy as np
import pytest

import helpers

ROOT = helpers.ROOT
STOCK = os.path.join(ROOT, "oracle", "_ref", "7z", "stock", "7zz")


def _stock_built():
    subprocess.check_call(["bash", os.path.join(ROOT, "oracle", "build_ref_7z.sh")])
    return os.path.exists(STOCK)


def _files(pkg, n, seed=7):
    import random
    rng = random.Random(seed)
    g2 = pkg.corpus.g2(4 << 20).tobytes()
    files, names = [], []
    for i in range(n):
        size = rng.choice([0, 1, 100, 4096, 65536, 65536, 70000, 131072, 200000]) if i % 5 else rng.randrange(0, 300000)
        kind = i % 4
        if kind == 0:
            o = rng.randrange(0, len(g2) - size - 1); f = g2[o:o + size]
        elif kind == 1:
            f = pkg.corpus.entropy_class(1 + (i % 3), size).tobytes() if size else b""
        elif kind == 2:
            f = bytes(size)
        else:
            f = (b"abcdefgh" * (size // 8 + 1))[:size]
        files.append(f); names.append(f"dir{i % 7}/file_{i:05d}" + ("_äö€" if i % 11 == 0 else "") + ".bin")
    return files, names


def _check_archive(arc_bytes, files, names, tmp_path, shown="ZSTD:v1.5,l3"):
    """what the stock 7zz says of the archive (recorded where it is not built): `t` passes, `l` lists every file with the method,
    `x` gives every file back"""
    def ask():
        arc = tmp_path / "a.7z"; arc.write_bytes(arc_bytes)
        out = subprocess.run([STOCK, "t", str(arc)], capture_output=True, text=True)
        tested = out.returncode == 0 and "Everything is Ok" in out.stdout
        lst = subprocess.run([STOCK, "l", "-slt", str(arc)], capture_output=True, text=True).stdout
        method = any(l.startswith("Method = ") and shown in l for l in lst.splitlines())
        outdir = tmp_path / "x"; outdir.mkdir()
        out = subprocess.run([STOCK, "x", "-o" + str(outdir), str(arc)], capture_output=True, text=True)
        extracted = out.returncode == 0 and all((outdir / n).is_file() for n in names)
        got = "".join(helpers.digest((outdir / n).read_bytes()) for n in names) if extracted else ""
        return tested, lst.count("Path = dir"), method, extracted, helpers.digest(got.encode())
    r = helpers.reference_answer("7zz_t_l_x", (arc_bytes, shown, *names), ask, _stock_built())
    assert r == (True, len(files), True, True, helpers.digest("".join(helpers.digest(f) for f in files).encode())), r


def test_container_writer_on_oracle_frames(pkg, tmp_path):
    files, names = _files(pkg, 60)
    L = pkg.load_library()
    packed = [helpers.oracle_compress(f, frameLog=17, windowLog=17, flags=1) if f else b"" for f in files]
    blob = np.frombuffer(b"".join(packed) or b"\0", dtype=np.uint8)
    pack = np.array([len(p) for p in packed], dtype=np.uint64); unpack = np.array([len(f) for f in files], dtype=np.uint64)
    crcs = np.array([zlib.crc32(f) for f in files], dtype=np.uint32)
    enc = [n.encode("utf-8") for n in names]; arr = (ctypes.c_char_p * len(enc))(*enc)
    mt = np.full(len(files), 132_000_000_000_000_000, dtype=np.uint64)
    cap = 32 + len(blob) + 100 * len(files) + sum(len(e) for e in enc) * 2 + 1024
    out = np.zeros(cap, dtype=np.uint8); n = ctypes.c_size_t()
    rc = L.b200z_7z_build_archive(blob.ctypes.data, pack.ctypes.data, unpack.ctypes.data, crcs.ctypes.data, arr, mt.ctypes.data, len(files), 3,
                                  out.ctypes.data, cap, ctypes.byref(n))
    assert rc == 0
    assert out[:6].tobytes() == b"7z\xbc\xaf\x27\x1c"
    _check_archive(out[:n.value].tobytes(), files, names, tmp_path)
    # too small a destination is refused, nothing is written past it
    assert L.b200z_7z_build_archive(blob.ctypes.data, pack.ctypes.data, unpack.ctypes.data, crcs.ctypes.data, arr, None, len(files), 3, out.ctypes.data, 100, ctypes.byref(n)) == -4


@pytest.mark.gpu
def test_one_call_archive_of_many_files(pkg, codec, tmp_path):
    """cfg5 shape in small: 3 000 mixed-entropy files around 64 KiB -> one GPU pass -> a .7z the stock reference verifies and extracts;
    per-file CRC32s come from the GPU (a wrong one fails `7zz t`)"""
    files, names = _files(pkg, 3000, seed=5)
    arc = codec.write_7z(files, names)
    _check_archive(arc, files, names, tmp_path)
    # the packed streams are the batch API's: file i compressed alone with 128 KiB frames
    parts, _ = codec.compress_batch(files[:50])
    pos = 32
    for p in parts:
        assert arc[pos:pos + len(p)] == p; pos += len(p)
