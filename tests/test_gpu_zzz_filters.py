"""GPU: Delta and the stateless branch converters through the C ABI (csrc/b2z_filter.cu) against the oracle and the
reference's own functions (their recorded answers where oracle/_ref is not built).  Sorts last: first hardware run of these
kernels (written after the round's GPU budget was spent; their sources are checked through the host emulation in tests/test_filters.py)."""
import numpy as np
import pytest

import helpers as H
from test_filters import ARM, ARM64, ARMT, DELTA, PPC, SPARC, X86, instruction_soup, oracle_filter, ref_filter, x86_soup

pytestmark = pytest.mark.gpu


def test_branch_converters(pkg, codec):
    for method in (ARM64, ARM, PPC, SPARC, ARMT):
        data = instruction_soup(method, 1_000_000, 21) + b"\x01\x02\x03"
        for prop in (0, 0x00ABC000):
            enc = codec.filter(method, True, data, prop)
            assert enc == oracle_filter(method, 1, data, prop), hex(method)
            assert H.digest(enc) == ref_filter(method, 1, data, prop)
            assert codec.filter(method, False, enc, prop) == data
    with pytest.raises(pkg.B200zError) as e:
        codec.filter(0x0303011B, True, b"\xe8" * 64, 0)              # BCJ2: four streams + a range coder, left to the host
    assert e.value.code == -6
    with pytest.raises(pkg.B200zError):
        codec.filter(ARM64, True, bytes(64), 2)                       # start offset must be a multiple of 4 (BranchMisc.cpp:57)


def test_x86_bcj(pkg, codec):
    for dens in (0.01, 0.2, 0.6):
        data = x86_soup(3_000_003, dens, 31)
        for pc in (0, 0x00400000):
            enc = codec.filter(X86, True, data, pc)
            assert enc == oracle_filter(X86, 1, data, pc), dens
            assert H.digest(enc) == ref_filter(X86, 1, data, pc)
            assert codec.filter(X86, False, enc, pc) == data
    for n in (0, 1, 4, 5, 6):
        d = b"\xe8\x01\x02\x03\x00\xe8"[:n]
        assert codec.filter(X86, True, d, 0) == oracle_filter(X86, 1, d, 0)


def test_delta(pkg, codec):
    data = pkg.corpus.entropy_class(2, 3_000_001).tobytes() + bytes(range(256)) * 100
    for dist in (1, 2, 4, 255, 256):
        enc = codec.filter(DELTA, True, data, dist)
        assert enc == oracle_filter(DELTA, 1, data, dist), dist
        assert codec.filter(DELTA, False, enc, dist) == data, dist
        assert H.digest(codec.filter(DELTA, False, data, dist)) == ref_filter(DELTA, 0, data, dist)
    assert codec.filter(DELTA, True, b"", 1) == b"" and codec.filter(DELTA, False, b"abc", 7) == b"abc"
