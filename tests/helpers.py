"""Test-side access to the checker libraries: oracle/liboracle.so (our C restatement) and
oracle/_ref/libref_zstd.so (the unmodified reference, compiled by oracle/Makefile), and the recorded answers of the
reference (tests/golden/reference_answers.json) that stand in for it where it is not built."""
import ctypes
import hashlib
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAXSEQ = 32768
ANSWERS = os.path.join(ROOT, "tests", "golden", "reference_answers.json")


def digest(data) -> str:
    """short content digest of bytes (what the recorded answers hold instead of the reference's output)"""
    return hashlib.sha256(bytes(data)).hexdigest()[:16]


_answers = None


def _tuples(v):
    return tuple(_tuples(x) for x in v) if isinstance(v, (list, tuple)) else v


def reference_answer(question, parts, ask, built):
    """The reference's answer to `question` about the inputs `parts` (bytes, numbers, strings).

    Where the reference library is `built`, `ask()` computes it (a JSON value: digests, sizes, flags) and it must equal the answer
    recorded for the same inputs; with B2Z_RECORD_REFERENCE=1 new answers are added to tests/golden/reference_answers.json.
    Elsewhere the recorded answer is returned, so a build without the reference is still checked against it -- an input that
    was never put to the reference (our encoder's output changed, say) fails until it is recorded again where the reference is built."""
    global _answers
    if _answers is None:
        _answers = json.load(open(ANSWERS)) if os.path.exists(ANSWERS) else {}
    h = hashlib.sha256(question.encode())
    for p in parts:
        h.update(b"\0" + (bytes(p) if isinstance(p, (bytes, bytearray, memoryview)) else repr(p).encode()))
    key = f"{question}:{h.hexdigest()[:16]}"
    if not built:
        assert key in _answers, f"no recorded answer of the reference for {key}: record it with B2Z_RECORD_REFERENCE=1 where oracle/_ref is built"
        return _tuples(_answers[key])
    got = json.loads(json.dumps(ask()))
    if key in _answers:
        assert _answers[key] == got, (key, _answers[key], got)
    elif os.environ.get("B2Z_RECORD_REFERENCE") == "1":
        _answers[key] = got
        import fcntl
        with open(ANSWERS, "a+") as f:                              # pytest-xdist workers record side by side
            fcntl.flock(f, fcntl.LOCK_EX)
            f.seek(0)
            text = f.read()
            table = json.loads(text) if text else {}
            table[key] = got
            f.seek(0); f.truncate()
            json.dump(table, f, indent=0, sort_keys=True)
    return _tuples(got)


def seq_fields(s):
    """(offBase, litLength, matchLength) of one packed sequence record (b2z_params.h B2Z_PACK_SEQ)"""
    s = int(s)
    return s & 0xFFFFFFF, (s >> 28) & 0x3FFFF, (s >> 46) & 0x3FFFF


class EncParams(ctypes.Structure):
    _fields_ = [(n, ctypes.c_uint32) for n in ("frameLog", "hashLogL", "hashLogS", "windowLog", "chunkLog", "flags", "regionLog", "ldmLog")]


_oracle = None
_ref = None


def oracle():
    global _oracle
    if _oracle is None:
        path = os.path.join(ROOT, "oracle", "liboracle.so")
        import subprocess
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "oracle"])     # no-op when up to date; never a stale checker
        O = ctypes.CDLL(path)
        O.b2zo_zstd_decompress.restype = ctypes.c_int64
        O.b2zo_zstd_decompress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t]
        O.b2zo_zstd_compress.restype = ctypes.c_int64
        O.b2zo_zstd_compress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(EncParams)]
        O.b2zo_zstd_compress_bound.restype = ctypes.c_size_t
        O.b2zo_zstd_compress_bound.argtypes = [ctypes.c_size_t, ctypes.POINTER(EncParams)]
        O.b2zo_zstd_find_sequences.restype = ctypes.c_int64
        O.b2zo_zstd_find_sequences.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(EncParams)] + [ctypes.c_void_p] * 4
        O.b2zo_xxh64.restype = ctypes.c_uint64
        O.b2zo_xxh64.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint64]
        _oracle = O
    return _oracle


def ref_available():
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_zstd.so"))


def ref():
    global _ref
    if _ref is None:
        Z = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_zstd.so"))
        Z.ZSTD_compressBound.restype = ctypes.c_size_t; Z.ZSTD_compressBound.argtypes = [ctypes.c_size_t]
        Z.ZSTD_createCCtx.restype = ctypes.c_void_p
        Z.ZSTD_freeCCtx.argtypes = [ctypes.c_void_p]
        Z.ZSTD_CCtx_setParameter.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]; Z.ZSTD_CCtx_setParameter.restype = ctypes.c_size_t
        Z.ZSTD_compress2.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t]; Z.ZSTD_compress2.restype = ctypes.c_size_t
        Z.ZSTD_decompress.restype = ctypes.c_size_t; Z.ZSTD_decompress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t]
        Z.ZSTD_isError.argtypes = [ctypes.c_size_t]
        Z.ZSTD_getErrorName.restype = ctypes.c_char_p; Z.ZSTD_getErrorName.argtypes = [ctypes.c_size_t]
        _ref = Z
    return _ref


def _np(data):
    return np.frombuffer(data, dtype=np.uint8) if len(data) else np.zeros(1, dtype=np.uint8)


def enc_params(**kw):
    p = EncParams()
    oracle().b2zo_enc_default_params(ctypes.byref(p), 3)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def oracle_compress(data, **kw) -> bytes:
    p = enc_params(**kw)
    src = _np(data)
    out = np.empty(oracle().b2zo_zstd_compress_bound(len(data), ctypes.byref(p)), dtype=np.uint8)
    r = oracle().b2zo_zstd_compress(out.ctypes.data, out.size, src.ctypes.data, len(data), ctypes.byref(p))
    assert r > 0, r
    return out[:r].tobytes()


def oracle_find_sequences(data, **kw):
    p = enc_params(**kw)
    src = _np(data); n = len(data)
    nblk = (n + 131071) // 131072
    seqs = np.zeros(nblk * MAXSEQ, dtype=np.uint64)
    nseq = np.zeros(nblk, dtype=np.uint32); nlit = np.zeros(nblk, dtype=np.uint32)
    lits = np.zeros(max(n, 1), dtype=np.uint8)
    r = oracle().b2zo_zstd_find_sequences(src.ctypes.data, n, ctypes.byref(p), seqs.ctypes.data, nseq.ctypes.data, lits.ctypes.data, nlit.ctypes.data)
    assert r == nblk
    return seqs, nseq, lits[:n], nlit


def oracle_candidates(data, **kw):
    """stage F tap: one candidate word per input byte, frames back to back (b2zo_zstd_candidates per frame)"""
    p = enc_params(**kw)
    O = oracle()
    O.b2zo_zstd_candidates.restype = None
    O.b2zo_zstd_candidates.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.POINTER(EncParams), ctypes.c_void_p]
    src = _np(data); n = len(data); F = 1 << p.frameLog
    cand = np.zeros(max(n, 1), dtype=np.uint32)
    for f0 in range(0, n, F):
        O.b2zo_zstd_candidates(src.ctypes.data + f0, min(F, n - f0), ctypes.byref(p), cand.ctypes.data + 4 * f0)
    return cand[:n]


def far_copies(pkg, n, every, span, seed=3, mutate=0.001, back=None):
    """text (the G2 generator) with long-range redundancy: BASELINE configs[2]'s recipe (corpus.inject_far_copies) at a test's scale"""
    d = pkg.corpus.g2(n)
    pkg.corpus.inject_far_copies(d, every=every, span=span, back=back, mutate=mutate, seed=seed)
    return d.tobytes()


def oracle_decompress(comp, n) -> bytes:
    dst = np.empty(n + 1, dtype=np.uint8); src = _np(comp)
    r = oracle().b2zo_zstd_decompress(dst.ctypes.data, n, src.ctypes.data, len(comp))
    if r < 0:
        raise ValueError(f"oracle decoder error {r}")
    return dst[:r].tobytes()


def ref_compress(data, level=3, checksum=0, **kw) -> bytes:
    Z = ref()
    c = Z.ZSTD_createCCtx()
    Z.ZSTD_CCtx_setParameter(c, 100, level); Z.ZSTD_CCtx_setParameter(c, 201, checksum)
    ids = dict(windowLog=101, hashLog=102, chainLog=103, searchLog=104, minMatch=105, targetLength=106, strategy=107,
               nbWorkers=400, enableLongDistanceMatching=160, contentSizeFlag=200)
    for k, v in kw.items():
        Z.ZSTD_CCtx_setParameter(c, ids[k], v)
    src = _np(data)
    out = np.empty(Z.ZSTD_compressBound(len(data)), dtype=np.uint8)
    r = Z.ZSTD_compress2(c, out.ctypes.data, out.size, src.ctypes.data, len(data))
    Z.ZSTD_freeCCtx(c)
    assert not Z.ZSTD_isError(r), Z.ZSTD_getErrorName(r)
    return out[:r].tobytes()


def ref_decompress(comp, n) -> bytes:
    Z = ref()
    dst = np.empty(n + 1, dtype=np.uint8); src = _np(comp)
    r = Z.ZSTD_decompress(dst.ctypes.data, n + 1, src.ctypes.data, len(comp))
    if Z.ZSTD_isError(r):
        raise ValueError(Z.ZSTD_getErrorName(r).decode())
    return dst[:r].tobytes()


def ref_zstd_result(comp, n):
    """digest of what the reference decoder makes of `comp` (at most n bytes), or "error" (recorded where the reference is absent)"""
    def ask():
        try:
            return digest(ref_decompress(comp, n))
        except ValueError:
            return "error"
    return reference_answer("zstd_decode", (comp, n), ask, ref_available())


def ref_size(coder, data, *args, **kw):
    """size of the reference encoder's output for `data` (coder: ref_compress, ref_lzma2_compress or ref_fl2_compress)"""
    def ask():
        out = coder(data, *args, **kw)
        return len(out if isinstance(out, bytes) else out[1])
    return reference_answer(f"{coder.__name__}_size", (data, args, sorted(kw.items())), ask,
                            ref_available() if coder is ref_compress else ref_lzma_available())


def sample_inputs(pkg, big=False):
    """name -> bytes: the seeded inputs shared by the CPU and GPU tests (edge cases included)."""
    g2 = pkg.corpus.g2
    cls = pkg.corpus.entropy_class
    d = {
        "empty": b"", "one": b"a", "tiny": b"hello hello hello hello", "seven": b"1234567", "eight": b"12345678",
        "g2_100k": g2(100_000).tobytes(),
        "g2_128k": g2(131072).tobytes(),
        "g2_128k+1": g2(131073).tobytes(),
        "g2_1m": g2(1 << 20).tobytes(),
        "noise": cls(1, 300_000).tobytes(), "skew": cls(2, 700_000).tobytes(), "tile": cls(3, 900_000).tobytes(),
        "zeros": bytes(500_000), "ones_33": b"\x01" * 33,
        "payload": b"TEST\n" + b" " * 999990 + b"\nEND.",       # the reference's regression payload (tests/regression.test:181)
        "mixed": g2(200_000).tobytes() + bytes(150_000) + cls(1, 100_000).tobytes() + cls(3, 250_000).tobytes(),
    }
    if big:
        d["g2_9m"] = g2(9 * (1 << 20) + 4321).tobytes()           # 3 frames, ragged tail
    return d


# ---------------------------------------------------------------- LZMA2 (method 21) ----------------------------------------
_ref_lzma = None


def ref_lzma_available():
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_lzma.so"))


def ref_xz_available():
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_xz.so"))


class _LzmaEncProps(ctypes.Structure):      # C/LzmaEnc.h:13-39
    _fields_ = [("level", ctypes.c_int), ("dictSize", ctypes.c_uint32), ("lc", ctypes.c_int), ("lp", ctypes.c_int), ("pb", ctypes.c_int),
                ("algo", ctypes.c_int), ("fb", ctypes.c_int), ("btMode", ctypes.c_int), ("numHashBytes", ctypes.c_int),
                ("numHashOutBits", ctypes.c_uint), ("mc", ctypes.c_uint32), ("writeEndMark", ctypes.c_uint), ("numThreads", ctypes.c_int),
                ("affinityGroup", ctypes.c_int32), ("reduceSize", ctypes.c_uint64), ("affinity", ctypes.c_uint64), ("affinityInGroup", ctypes.c_uint64)]


class _Lzma2EncProps(ctypes.Structure):     # C/Lzma2Enc.h:15-23
    _fields_ = [("lzmaProps", _LzmaEncProps), ("blockSize", ctypes.c_uint64), ("numBlockThreads_Reduced", ctypes.c_int),
                ("numBlockThreads_Max", ctypes.c_int), ("numTotalThreads", ctypes.c_int), ("numThreadGroups", ctypes.c_uint)]


def ref_lzma():
    global _ref_lzma
    if _ref_lzma is None:
        L = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_lzma.so"))
        L.FL2_compressBound.restype = ctypes.c_size_t; L.FL2_compressBound.argtypes = [ctypes.c_size_t]
        L.FL2_compressMt.restype = ctypes.c_size_t
        L.FL2_compressMt.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_uint]
        L.Lzma2Decode.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p, ctypes.POINTER(ctypes.c_size_t),
                                  ctypes.c_ubyte, ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.c_void_p]
        L.FL2_isError.argtypes = [ctypes.c_size_t]
        L.Lzma2Enc_Create.restype = ctypes.c_void_p; L.Lzma2Enc_Create.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.Lzma2Enc_Destroy.argtypes = [ctypes.c_void_p]
        L.Lzma2Enc_SetProps.argtypes = [ctypes.c_void_p, ctypes.POINTER(_Lzma2EncProps)]
        L.Lzma2Enc_WriteProperties.restype = ctypes.c_ubyte; L.Lzma2Enc_WriteProperties.argtypes = [ctypes.c_void_p]
        L.Lzma2Enc_Encode2.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
        L.Lzma2EncProps_Init.argtypes = [ctypes.POINTER(_Lzma2EncProps)]
        _ref_lzma = L
    return _ref_lzma


def ref_fl2_compress(data, level=5, threads=1):
    """reference Fast-LZMA2 encoder (C/fast-lzma2/fl2_compress.c) -> (dictProp, raw LZMA2 stream).
    FL2_compress prepends the 1-byte dictionary property (and may append a hash after the 0x00 end marker)."""
    L = ref_lzma(); src = _np(data)
    out = np.empty(L.FL2_compressBound(len(data)) + 64, dtype=np.uint8)
    r = L.FL2_compressMt(out.ctypes.data, out.size, src.ctypes.data, len(data), level, threads)
    assert not L.FL2_isError(r)
    return int(out[0]) & 0x3F, out[1:r].tobytes()


def ref_lzma2_compress(data, level=5, dict_size=0, lc=-1, lp=-1, pb=-1, block_size=0, threads=1):
    """reference stock LZMA2 encoder (C/Lzma2Enc.c) -> (dictProp, raw LZMA2 stream)."""
    L = ref_lzma(); src = _np(data)
    p = _Lzma2EncProps(); L.Lzma2EncProps_Init(ctypes.byref(p))
    p.lzmaProps.level = level; p.lzmaProps.dictSize = dict_size; p.lzmaProps.lc = lc; p.lzmaProps.lp = lp; p.lzmaProps.pb = pb
    p.blockSize = block_size; p.numTotalThreads = threads; p.numBlockThreads_Max = threads
    alloc = ctypes.c_void_p.in_dll(L, "g_Alloc"); big = ctypes.c_void_p.in_dll(L, "g_BigAlloc")
    h = L.Lzma2Enc_Create(ctypes.addressof(alloc), ctypes.addressof(big))
    assert h
    assert L.Lzma2Enc_SetProps(h, ctypes.byref(p)) == 0
    prop = L.Lzma2Enc_WriteProperties(h)
    out = np.empty(len(data) + len(data) // 3 + 4096, dtype=np.uint8); n = ctypes.c_size_t(out.size)
    rc = L.Lzma2Enc_Encode2(h, None, out.ctypes.data, ctypes.byref(n), None, src.ctypes.data, len(data), None)
    L.Lzma2Enc_Destroy(h)
    assert rc == 0, rc
    return int(prop), out[:n.value].tobytes()


def oracle_lzma2_decompress(comp, n, dict_prop):
    O = oracle()
    O.b2zo_lzma2_decompress.restype = ctypes.c_int64
    O.b2zo_lzma2_decompress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_void_p]
    dst = np.empty(n + 1, dtype=np.uint8); src = _np(comp); used = ctypes.c_size_t(0)
    r = O.b2zo_lzma2_decompress(dst.ctypes.data, n, src.ctypes.data, len(comp), dict_prop, ctypes.byref(used))
    if r < 0:
        raise ValueError(f"oracle lzma2 decoder error {r}")
    return dst[:r].tobytes(), used.value


def ref_lzma2_decompress(comp, n, dict_prop):
    """reference decoder, one-call form (C/Lzma2Dec.c: Lzma2Decode)."""
    L = ref_lzma(); src = _np(comp); dst = np.empty(n + 1, dtype=np.uint8)
    dl = ctypes.c_size_t(n); sl = ctypes.c_size_t(len(comp)); st = ctypes.c_int(0)
    alloc = ctypes.c_void_p.in_dll(L, "g_Alloc")
    rc = L.Lzma2Decode(dst.ctypes.data, ctypes.byref(dl), src.ctypes.data, ctypes.byref(sl), dict_prop, 1, ctypes.byref(st), ctypes.addressof(alloc))
    if rc != 0:
        raise ValueError(f"reference lzma2 decoder error {rc}")
    return dst[:dl.value].tobytes(), sl.value


def ref_lzma2_result(comp, n, dict_prop):
    """(digest of the output, bytes consumed) of the reference LZMA2 decoder on `comp`, or None where it reports an error"""
    def ask():
        try:
            out, used = ref_lzma2_decompress(comp, n, dict_prop)
        except ValueError:
            return None
        return digest(out), used
    return reference_answer("lzma2_decode", (comp, n, dict_prop), ask, ref_lzma_available())


def lzma2_result(out_used):
    """(bytes, consumed) of a decoder in the form ref_lzma2_result answers"""
    return None if out_used is None else (digest(out_used[0]), out_used[1])


def oracle_lzma2_compress(data, **kw):
    """sequential statement of the GPU LZMA2 encoder -> (dictProp, raw LZMA2 stream)"""
    O = oracle(); p = enc_params(**kw); src = _np(data)
    O.b2zo_lzma2_compress_bound.restype = ctypes.c_size_t; O.b2zo_lzma2_compress_bound.argtypes = [ctypes.c_size_t, ctypes.POINTER(EncParams)]
    O.b2zo_lzma2_compress.restype = ctypes.c_int64
    O.b2zo_lzma2_compress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(EncParams), ctypes.POINTER(ctypes.c_uint32)]
    out = np.empty(O.b2zo_lzma2_compress_bound(len(data), ctypes.byref(p)), dtype=np.uint8); prop = ctypes.c_uint32(0)
    r = O.b2zo_lzma2_compress(out.ctypes.data, out.size, src.ctypes.data, len(data), ctypes.byref(p), ctypes.byref(prop))
    assert r > 0, r
    return prop.value, out[:r].tobytes()


def ref_lzma2_decompress_mt(comp, n, dict_prop, threads):
    """the reference's MT decoder path (C/Lzma2DecMt.c driven as Lzma2Decoder.cpp:95-186 does) -> (bytes, ran_multithreaded)"""
    L = ref_lzma(); src = _np(comp); dst = np.empty(n + 1, dtype=np.uint8)
    L.refh_lzma2_decode_mt.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p, ctypes.c_size_t,
                                       ctypes.c_uint, ctypes.c_uint, ctypes.POINTER(ctypes.c_int)]
    out = ctypes.c_size_t(0); mt = ctypes.c_int(0)
    rc = L.refh_lzma2_decode_mt(dst.ctypes.data, n, ctypes.byref(out), src.ctypes.data, len(comp), dict_prop, threads, ctypes.byref(mt))
    if rc != 0:
        raise ValueError(f"reference lzma2 MT decoder error {rc}")
    return dst[:out.value].tobytes(), bool(mt.value)


def ref_lzma2_mt_result(comp, n, dict_prop, threads):
    """(digest of the output, ran multithreaded) of the reference's MT decoder path"""
    def ask():
        out, mt = ref_lzma2_decompress_mt(comp, n, dict_prop, threads)
        return digest(out), mt
    return reference_answer("lzma2_decode_mt", (comp, n, dict_prop, threads), ask, ref_lzma_available())


# ---------------------------------------------------------------- host emulation of the kernel sources (tests/cuemu)
def cuemu_library():
    """builds and loads tests/cuemu/libcuemu_kernels.so; with B2Z_CUEMU_ASAN=1 the AddressSanitizer variant (run pytest with
    LD_PRELOAD=$(/usr/bin/gcc -print-file-name=libasan.so) ASAN_OPTIONS=detect_leaks=0:detect_stack_use_after_return=0)"""
    import subprocess
    d = os.path.join(ROOT, "tests", "cuemu")
    name = ("libcuemu_kernels_asan.so" if os.environ.get("B2Z_CUEMU_ASAN") else
            "libcuemu_kernels_ubsan.so" if os.environ.get("B2Z_CUEMU_UBSAN") else "libcuemu_kernels.so")     # UBSan: LD_PRELOAD libubsan.so, pytest -s
    import fcntl
    with open(os.path.join(d, ".build.lock"), "w") as lock:         # pytest-xdist workers would otherwise run make on the same target at once
        fcntl.flock(lock, fcntl.LOCK_EX)
        subprocess.check_call(["make", "-s", "-C", d, name])
    return ctypes.CDLL(os.path.join(d, name))


def capped_match_near_boundary(pkg):
    """a match of >= 255 bytes (stage C stores the capped length 255) that starts 100 bytes before a 128 KiB block / slice end and
    is not a repeat of the previous distance: the long-match path must clip it to the boundary (found by the emulator fuzz: the
    capped candidate used to be extended from byte 224 even when fewer bytes were left)"""
    noise = pkg.corpus.entropy_class(1, 131072 * 2 + 5000).tobytes()
    a = bytearray(noise)
    chunk = bytes(a[1000:5000])
    a[131072 - 100:131072 - 100 + 4000] = chunk                     # second copy straddles the boundary at 131072
    a[131072 + 60_000:131072 + 60_000 + 300] = chunk[:300]          # and one whose whole length (300 > 255) fits: the extension proper
    return bytes(a)
