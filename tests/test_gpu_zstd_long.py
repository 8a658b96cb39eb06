"""GPU: the long mode of the Zstandard encoder (B200Z_P_LONG; the reference's long=N, ZstdEncoder.cpp:128-146 / zstd_ldm.c) through the
C ABI: stage F per 1 MiB region + stage L per frame == the oracle byte for byte; frames of up to 128 MiB decode with the reference's
decoder and with the engine's own; BASELINE configs[2]'s recipe (far copies with mutations) is where it pays."""
import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu


def test_long_mode_equals_the_oracle(pkg):
    n = (40 << 20) + 4321
    data = helpers.far_copies(pkg, n, every=4 << 20, span=(256 << 10, 1 << 20))
    c = pkg.Codec(0, long=24)
    assert c.get("long") == 24 and c.get("frame_log") == 27 and c.get("window_log") == 24     # frames of 8 windows
    p = dict(frameLog=27, windowLog=24, regionLog=20, ldmLog=18)
    assert np.array_equal(c.stage_f(data), helpers.oracle_candidates(data, **p))          # stage F per region, then stage L
    comp = c.compress(data)
    assert comp == helpers.oracle_compress(data, **p)
    assert c.decompress(comp, n) == data
    assert helpers.ref_zstd_result(comp, n) == helpers.digest(data)
    plain = pkg.Codec(0)
    assert len(comp) < len(plain.compress(data)) - 1_000_000                               # ~9 spans of ~600 KiB found again
    # the level does not change the long mode's parse (the price-based stage C + Z works on frames of <= 16 MiB)
    c19 = pkg.Codec(0, level=19, long=24)
    assert c19.compress(data) == comp
    # leaving the mode: 1 MiB frames again
    c.set("long", 0)
    assert c.get("frame_log") == 20 and c.compress(data) == plain.compress(data)
    c.close(); c19.close(); plain.close()


def test_window_of_128_mib(pkg):
    """long=27 on 300 MiB: one frame, window 2^27; the engine's decoder (units of 8 blocks, far matches wait for the unit that wrote
    their source) and the reference's (default window limit 2^27) give the input back; equal to the oracle byte for byte; copies
    planted up to 128 MiB back are found (the stream is smaller than the plain one by most of their size)"""
    n = (300 << 20) + 99
    data = helpers.far_copies(pkg, n, every=32 << 20, span=(1 << 20, 4 << 20), seed=3, back=128 << 20)
    c = pkg.Codec(0, long=27)
    comp = c.compress(data)
    assert comp[12:16] == b"\x28\xb5\x2f\xfd" and 10 + (comp[17] >> 3) == 27 and int.from_bytes(comp[18:22], "little") == n
    assert c.decompress(comp, n) == data
    assert helpers.ref_zstd_result(comp, n) == helpers.digest(data)
    plain = pkg.Codec(0)
    assert len(comp) < len(plain.compress(data)) - 6_000_000                               # 9 spans of ~2.5 MiB, at a ratio of 2.4
    assert comp == helpers.oracle_compress(data, frameLog=30, windowLog=27, regionLog=20, ldmLog=21)
    c.close(); plain.close()


def test_long_mode_over_the_devices_of_a_group(pkg):
    """device count is invisible in the long mode too: batches of whole frames are dealt over the devices"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one device")
    n = (600 << 20) + 5
    data = helpers.far_copies(pkg, n, every=8 << 20, span=(1 << 20, 2 << 20), seed=9, back=16 << 20)
    one = pkg.Codec(0, long=24); two = pkg.Codec(devices=[0, 1], long=24)                   # frames of 128 MiB: five of them, dealt in batches of 256 MiB
    a = one.compress(data); b = two.compress(data)
    assert a == b and two.decompress(b, n) == data
    one.close(); two.close()
