"""CPU: the long mode of the Zstandard encoder as the oracle states it (oracle/zstd_enc_oracle.c: regions for stage F, ldm_frame for
stage L) -- the restatement of the reference's long=N (ZstdEncoder.cpp:128-146, 322-331 -> ZSTD_c_enableLongDistanceMatching, zstd_ldm.c):
frames stay format-valid for the reference's decoder, far copies are found, and the gain is close to what the reference's own
long-distance matcher gets on the same bytes."""
import numpy as np
import pytest

import helpers as H


def _frames(comp):
    """(windowLog byte, content size) of every zstd frame of a stream of [skippable hint][frame] pairs"""
    out = []; i = 0
    while i < len(comp):
        if comp[i:i + 4] == b"\x50\x2a\x4d\x18":
            i += 12; continue
        assert comp[i:i + 4] == b"\x28\xb5\x2f\xfd"
        out.append((10 + (comp[i + 5] >> 3), int.from_bytes(comp[i + 6:i + 10], "little"), i))
        # the size hint in front of the frame gives its length
        hint = int.from_bytes(comp[i - 4:i], "little")
        i += hint
    return out


def test_long_mode_finds_far_copies_and_stays_valid(pkg):
    n = (24 << 20) + 777
    data = H.far_copies(pkg, n, every=4 << 20, span=(256 << 10, 1 << 20))
    plain = H.oracle_compress(data)
    long_ = H.oracle_compress(data, frameLog=28, windowLog=25, regionLog=20, ldmLog=19)      # what B200Z_P_LONG 25 sets
    assert H.oracle_decompress(long_, n) == data
    fr = _frames(long_)
    assert [(w, s) for w, s, _ in fr] == [(25, n)]                             # one frame (of up to 8 windows), window 2^25
    gain = len(plain) - len(long_)
    assert gain > 1_000_000
    assert H.ref_zstd_result(long_, n) == H.digest(data)
    ref_gain = H.ref_size(H.ref_compress, data, level=3) - H.ref_size(H.ref_compress, data, level=3, windowLog=25, enableLongDistanceMatching=1)
    assert gain > 0.9 * ref_gain, (gain, ref_gain)                          # measured: 1.49 MB against the reference's 1.55 MB


def test_long_mode_without_far_copies_changes_little(pkg):
    """no long-range redundancy: stage L finds (next to) nothing, and regions cost nothing against frames of the same size"""
    data = pkg.corpus.g2(6 << 20).tobytes()
    plain = H.oracle_compress(data, regionLog=20)
    long_ = H.oracle_compress(data, frameLog=23, windowLog=23, regionLog=20, ldmLog=16)
    assert H.oracle_decompress(long_, len(data)) == data
    assert abs(len(long_) - len(plain)) < len(plain) // 500
    # a frame of one region is the frame of an encoder without regions
    assert H.oracle_compress(data[:1 << 20], frameLog=20, windowLog=20, regionLog=20, ldmLog=13) == H.oracle_compress(data[:1 << 20], regionLog=0)


def test_window_of_128_mib(pkg):
    """long=27: window 2^27 in a frame of up to 1 GiB; copies planted up to 128 MiB back are coded as matches (offsets beyond
    64 MiB appear, none beyond the window), and the reference decodes the stream with its default window limit (2^27)"""
    n = (1 << 27) + (41 << 20) + 12345
    data = H.far_copies(pkg, n, every=16 << 20, span=(1 << 20, 2 << 20), seed=5, back=128 << 20)
    p = dict(frameLog=30, windowLog=27, regionLog=20, ldmLog=21)
    comp = H.oracle_compress(data, **p)
    fr = _frames(comp)
    assert [(w, s) for w, s, _ in fr] == [(27, n)]
    seqs, nseq, lits, nlit = H.oracle_find_sequences(data, **p)
    far = 0; top = 0
    for b in range(len(nseq)):
        ob = seqs[b * H.MAXSEQ:b * H.MAXSEQ + int(nseq[b])] & np.uint64(0xFFFFFFF)
        far += int((ob > (64 << 20) + 3).sum()); top = max(top, int(ob.max()) if len(ob) else 0)
    assert far > 10 and top - 3 < (1 << 27)
    assert H.oracle_decompress(comp, n) == data
    assert H.ref_zstd_result(comp, n) == H.digest(data)
    plain = H.oracle_compress(data[:32 << 20])
    assert len(comp) < len(plain) * (n / (32 << 20)) * 0.97                    # 10 spans of 1-2 MiB in 169 MiB: some 4 % less than without
