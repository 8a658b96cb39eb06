"""GPU parity tests of the zstd encoder path (through the C ABI in include/b200z.h).

Parity bar (north_star): frames are format-valid and the reference's own decoder
(oracle/_ref, built from /root/reference/C/zstd) round-trips them to identical bytes; in
addition the CUDA path must equal the oracle restatement byte for byte (integer algorithm).
"""
import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def inputs(pkg):
    return helpers.sample_inputs(pkg, big=True)


def test_stage_f_matches_oracle(pkg, codec, inputs):
    """stage F tap (one candidate word per position) == oracle b2zo_zstd_candidates, default and non-default chunk sizes / table logs."""
    for name in ("g2_1m", "tile", "zeros", "mixed", "g2_128k+1", "skew", "g2_9m", "seven", "eight"):
        data = inputs[name]
        assert np.array_equal(codec.stage_f(data), helpers.oracle_candidates(data)), name
    data = inputs["mixed"] + inputs["g2_1m"]
    for cl, hl, hs, fl in ((5, 15, 14, 18), (6, 12, 13, 20), (8, 14, 15, 19), (7, 15, 14, 17)):
        c = pkg.Codec(0, frame_log=fl, chunk_log=cl, hash_log_l=10, hash_log_s=hs)
        c.set("hash_log_l", hl)
        assert np.array_equal(c.stage_f(data), helpers.oracle_candidates(data, frameLog=fl, windowLog=fl, chunkLog=cl, hashLogL=hl, hashLogS=hs)), (cl, hl, hs, fl)
        c.close()


def test_stage_m_matches_oracle(pkg, codec, inputs):
    """stage F + stage G taps (final sequences + literals per block) == oracle find_sequences."""
    for name in ("g2_1m", "tile", "zeros", "mixed", "g2_128k+1", "skew", "g2_9m"):
        data = inputs[name]
        seqs, nseq, lits, nlit = codec.stage_m(data)
        oseqs, onseq, olits, onlit = helpers.oracle_find_sequences(data)
        assert np.array_equal(nseq, onseq), (name, nseq[:8], onseq[:8])
        assert np.array_equal(nlit, onlit), (name, nlit[:8], onlit[:8])
        for b in range(len(nseq)):
            s = slice(b * helpers.MAXSEQ, b * helpers.MAXSEQ + int(nseq[b]))
            if not np.array_equal(seqs[s], oseqs[s]):
                i = int(np.nonzero(seqs[s] != oseqs[s])[0][0])
                raise AssertionError(f"{name}: block {b} seq {i}: gpu {int(seqs[s][i]):#x} oracle {int(oseqs[s][i]):#x}")
            l = slice(b * 131072, b * 131072 + int(nlit[b]))
            assert np.array_equal(lits[l], olits[l]), (name, b)


def test_frames_equal_oracle_and_roundtrip(pkg, codec, inputs):
    for name, data in inputs.items():
        comp = codec.compress(data)
        want = helpers.oracle_compress(data)
        if comp != want:
            n = min(len(comp), len(want))
            i = next((k for k in range(n) if comp[k] != want[k]), n)
            raise AssertionError(f"{name}: frame bytes differ from oracle at {i} (sizes {len(comp)} vs {len(want)})")
        assert helpers.oracle_decompress(comp, len(data)) == data, name
        assert helpers.ref_zstd_result(comp, len(data)) == helpers.digest(data), name


def test_params_and_hints(pkg, inputs):
    """non-default geometry and the skippable size hints stay byte-identical to the oracle and decodable."""
    data = inputs["g2_9m"][: 3 * (1 << 20) + 77]
    c = pkg.Codec(0, frame_log=19, chunk_log=6, hash_log_s=13, flags=1)
    comp = c.compress(data)
    assert comp == helpers.oracle_compress(data, frameLog=19, windowLog=19, chunkLog=6, hashLogS=13, flags=1)
    assert comp[:4] == b"\x50\x2a\x4d\x18"
    assert helpers.ref_zstd_result(comp, len(data)) == helpers.digest(data)
    c.close()


def test_ratio_vs_reference_level3(pkg, codec):
    """ratio within 1 % of the reference's level 3 on the BASELINE cfg2 text shape (16 MiB sample)."""
    data = pkg.corpus.g2(16 << 20).tobytes()
    ours = len(codec.compress(data)); ref = helpers.ref_size(helpers.ref_compress, data, 3)
    assert ours <= ref * 1.01, (ours, ref)


def test_device_resident_and_stats(pkg, codec):
    import torch
    data = pkg.corpus.g2(8 << 20)
    src = torch.from_numpy(data).cuda()
    dst = torch.empty(codec.compress_bound(src.numel()), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    codec.reset_stats()
    n = codec.compress_device(src.data_ptr(), src.numel(), dst.data_ptr(), dst.numel())
    comp = dst[:n].cpu().numpy().tobytes()
    assert comp == helpers.oracle_compress(data.tobytes())
    assert codec.stat(6) >= 4 and codec.stat(1) > 0 and codec.stat(2) > 0


def test_bad_arguments(pkg, codec):
    with pytest.raises(pkg.B200zError):
        codec.set("frame_log", 40)
    import ctypes
    sz = ctypes.c_size_t()
    buf = np.zeros(64, dtype=np.uint8)
    rc = pkg.load_library().b200z_zstd_compress_host(codec.h, buf.ctypes.data, 64, buf.ctypes.data, 8, ctypes.byref(sz))
    assert rc == -4


def test_device_batches_are_invisible(pkg):
    """inputs larger than one kernel batch are compressed batch after batch; the bytes do not depend on the batch size"""
    data = pkg.corpus.g2(21 * (1 << 20) + 3210).tobytes()
    c = pkg.Codec(0, batch_log=22)
    comp = c.compress(data)
    assert comp == helpers.oracle_compress(data)
    c.close()


def test_batch_of_files(codec, pkg):
    """Many independent files in one call (BASELINE configs[4] shape: mixed-entropy files around 64 KiB): each file's bytes
    equal compressing it alone with 128 KiB frames (oracle), the reference decoder restores each file on its own, and the
    concatenated output decodes to the files back to back."""
    import random
    rng = random.Random(11)
    g2 = pkg.corpus.g2(6 << 20).tobytes()
    files = []
    for i in range(150):
        n = rng.choice([0, 1, 7, 1000, 65536, 65536, 65536, 70000, 131072, 131073, 300000, rng.randrange(1, 200000)])
        kind = i % 4
        if kind == 0:
            o = rng.randrange(0, len(g2) - n - 1); f = g2[o:o + n]
        elif kind == 1:
            f = pkg.corpus.entropy_class(1 + (i % 3), n).tobytes() if n else b""
        elif kind == 2:
            f = bytes(n)
        else:
            f = (b"abcdefgh" * (n // 8 + 1))[:n]
        files.append(f)
    parts, whole = codec.compress_batch(files)
    assert b"".join(parts) == whole
    for i, (f, c) in enumerate(zip(files, parts)):
        if not f:
            assert c == b""
            continue
        assert c == helpers.oracle_compress(f, frameLog=17, windowLog=17, flags=1), i
        if i % 7 == 0:
            assert helpers.ref_zstd_result(c, len(f)) == helpers.digest(f)
    assert codec.decompress(whole, max_size=sum(map(len, files))) == b"".join(files)
    # several kernel batches (batch_log 22 = 32 frames per batch): same bytes
    c2 = pkg.Codec(0, batch_log=22)
    parts2, whole2 = c2.compress_batch(files)
    assert whole2 == whole and parts2 == parts
    c2.close()


def test_host_batches_and_device_count_are_invisible(pkg):
    """the host-pointer calls cut their input into batches of whole frames and deal them over the devices of the context: the bytes
    depend neither on the batch size nor on the number of devices (workers), and the decoder restores the input through the same
    dispatcher.  Runs with every GPU of the box; on one GPU the same device is listed three times (three workers, own streams and
    scratch each), which exercises the ordering logic all the same."""
    import torch
    data = pkg.corpus.g2(37 * (1 << 20) + 777).tobytes() + bytes(3 << 20) + pkg.corpus.entropy_class(1, 2_000_000).tobytes()
    want = helpers.oracle_compress(data)
    n = torch.cuda.device_count()
    groups = [[0], [0, 0, 0]] + ([list(range(2)), list(range(n))] if n >= 2 else [])
    for devs in groups:
        for hb in (22, 24, 30):
            c = pkg.Codec(devices=devs, host_batch_log=hb)
            comp = c.compress(data)
            assert comp == want, (devs, hb, len(comp), len(want))
            assert c.decompress(comp) == data, (devs, hb)
            c.close()


def test_more_than_4_gib_in_one_call(pkg):
    """4.5 GiB through one host-pointer compress and one decompress call: offsets past 2^32, several pipeline batches.  Frames are
    independent, so the first and the last frames must equal the oracle's frames of the same bytes; the whole must round-trip."""
    import torch
    n = (9 << 29) + 12345
    host = torch.empty(n, dtype=torch.uint8).pin_memory()
    pkg.corpus.g2_into(host.data_ptr(), n)
    c = pkg.Codec(0)
    bound = c.compress_bound(n)
    comp = torch.empty(bound, dtype=torch.uint8).pin_memory()
    m = c.compress_into(host.data_ptr(), n, comp.data_ptr(), bound)
    data = host.numpy()
    first = helpers.oracle_compress(data[:1 << 20].tobytes())
    assert comp[:len(first)].numpy().tobytes() == first
    tail_start = (n >> 20) << 20
    last = helpers.oracle_compress(data[tail_start:].tobytes())
    assert comp[m - len(last):m].numpy().tobytes() == last
    back = torch.empty(n, dtype=torch.uint8).pin_memory()
    assert c.decompress_into(comp.data_ptr(), m, back.data_ptr(), n) == n
    assert torch.equal(back, host)
    c.close()


def test_level_ladder_matches_oracle(pkg, inputs):
    """B200Z_P_LEVEL below the price-based levels selects stage F's rung (1-2: the short table alone; 3-4: both tables; 5-7: both +
    the lower lanes of a position's step): frames equal the oracle run with the same level's parameters, the reference decoder restores
    them"""
    import ctypes
    data = inputs["mixed"] + inputs["g2_1m"] + b"0123456789abcdef" * 5000
    sizes = {}
    for level in (1, 2, 3, 4, 5, 7):
        p = helpers.EncParams(); helpers.oracle().b2zo_enc_default_params(ctypes.byref(p), level)
        c = pkg.Codec(0, level=level)
        comp = c.compress(data)
        assert comp == helpers.oracle_compress(data, flags=p.flags, hashLogS=p.hashLogS), level
        assert helpers.ref_zstd_result(comp, len(data)) == helpers.digest(data), level
        sizes[level] = len(comp)
        c.close()
    assert sizes[1] == sizes[2] and sizes[3] == sizes[4] and sizes[5] == sizes[7]
    assert len({sizes[1], sizes[3], sizes[5]}) == 3, sizes           # three different finders (which one wins depends on the data: text 1 < 3 = 5, code 1 < 3 < 5)
