"""CPU: oracle/zstd_opt_oracle.c -- the price-based Zstandard parse (flag bit 5; stage C candidates + stage Z per-block dynamic
programme) writes valid frames (the reference decoder and the oracle decoder restore the input), its sequences are valid, and
the ratio reaches the reference's level-9..12 class at the same 1 MiB window."""
import numpy as np
import pytest

import helpers as H

ZOPT = 0x20


def test_roundtrip_reference_and_oracle_decoders(pkg):
    for name, data in H.sample_inputs(pkg, big=True).items():
        for flags in (1 | ZOPT, 3 | ZOPT):                     # size hints; + XXH64 content checksum
            comp = H.oracle_compress(data, flags=flags)
            assert H.oracle_decompress(comp, len(data)) == data, name
            assert H.ref_zstd_result(comp, len(data)) == H.digest(data), name


def test_sequences_are_valid_and_cover_every_block(pkg):
    data = pkg.corpus.g2((1 << 20) + 200_001).tobytes() + bytes(70_000) + pkg.corpus.entropy_class(3, 90_000).tobytes()
    n = len(data)
    seqs, nseq, lits, nlit = H.oracle_find_sequences(data, flags=1 | ZOPT)
    F = 1 << 20; blk = 0
    for f0 in range(0, n, F):
        fn = min(F, n - f0)
        for b0 in range(0, fn, 131072):
            bn = min(131072, fn - b0)
            rep = [0, 0, 0]; pos = 0; nl = 0
            for i in range(int(nseq[blk])):
                ob, ll, ml = H.seq_fields(seqs[blk * H.MAXSEQ + i])
                assert ml >= 3
                lit_bytes = bytes(lits[f0 + b0 + nl:f0 + b0 + nl + ll]); assert lit_bytes == data[f0 + b0 + pos:f0 + b0 + pos + ll]
                pos += ll; nl += ll
                if ob > 3:                                       # the decoder's offset history rules (RFC 8878 3.1.1.5)
                    off = ob - 3; rep = [off, rep[0], rep[1]]
                else:
                    idx = ob - 1 + (1 if ll == 0 else 0)
                    off = rep[0] - 1 if idx == 3 else rep[idx]
                    assert off > 0                               # a repcode never refers to history the block has not set itself
                    if idx == 1: rep = [off, rep[0], rep[2]]
                    elif idx >= 2: rep = [off, rep[0], rep[1]]
                src_pos = f0 + b0 + pos
                assert src_pos - off >= f0 and pos + ml <= bn
                assert all(data[src_pos + k] == data[src_pos + k - off] for k in range(0, ml, max(1, ml // 64)))
                pos += ml
            assert pos + (int(nlit[blk]) - nl) == bn               # trailing literals close the block
            assert bytes(lits[f0 + b0 + nl:f0 + b0 + int(nlit[blk])]) == data[f0 + b0 + pos:f0 + b0 + bn]
            blk += 1


def test_ratio_class(pkg):
    data = pkg.corpus.g2(8 << 20).tobytes(); n = len(data)
    l3 = len(H.oracle_compress(data))
    opt = len(H.oracle_compress(data, flags=1 | ZOPT))
    opt22 = len(H.oracle_compress(data, flags=1 | ZOPT, frameLog=22, windowLog=22))
    assert opt < 0.95 * l3 and opt22 < opt                      # measured 2.53 against 2.39; 4 MiB frames 2.61
    ref9 = H.ref_size(H.ref_compress, data, level=9, windowLog=20)
    ref16 = H.ref_size(H.ref_compress, data, level=16, windowLog=20)
    assert opt < ref9 and opt < 1.08 * ref16                # between the reference's level 9 and its level 16 (optimal parse on binary trees)
