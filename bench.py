#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 zstd hot path (BASELINE.json configs[1]).

One "step" = one pass of the hot path over one batch of synthetic input: zstd level-3 encode of
the rank's corpus shard followed by decode of the produced frames (round trip verified on the
device, outside the timed region).  Metric: MB/s of uncompressed data through encode+decode,
MB = 1e6 bytes:   value = units / (t_enc + t_dec).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--size-mib M] [--impl ours|reference]
  torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU, weak scaling)

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definitions.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--size-mib", type=int, default=4096, help="uncompressed MiB per GPU per step (cfg2: 4 GiB)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample-mib", type=int, default=4096, help="sample for the CPU reference arm (default: the GPU arm's 4 GiB, same config; ~7 s per pass on 128 threads)")
    ap.add_argument("--no-files-extra", action="store_true", help="skip extra.many_files_7z (BASELINE configs[4]: 100 000 files of 64 KiB -> one non-solid .7z, one GPU pass)")
    ap.add_argument("--no-lzma2-extra", action="store_true", help="skip extra.lzma2 (BASELINE configs[3] measured beside the zstd headline: method 21 as -m0=flzma2 -mx5 selects it)")
    ap.add_argument("--no-refstreams-extra", action="store_true", help="skip extra.reference_streams (reference-written single-frame zstd and stock LZMA2 streams through the engine's decoders)")
    ap.add_argument("--no-long-extra", action="store_true", help="skip extra.long_range (BASELINE configs[2]: 8 GiB of text with far copies, long=27)")
    ap.add_argument("--long-mib", type=int, default=8192, help="extra.long_range: MiB of G3 input (configs[2]: 8 GiB)")
    ap.add_argument("--codec", default="zstd", choices=["zstd", "lzma2"],
                    help="zstd: method 4F71101 level 3 (the headline, BASELINE configs[1]); lzma2: method 21 (configs[3])")
    ap.add_argument("--level", type=int, default=3, help="--codec zstd: B200Z_P_LEVEL (1-7 stage M, the measured headline; 8-22 the price-based stage C + stage Z)")
    ap.add_argument("--lzma2-parse", type=int, default=1, choices=[0, 1],
                    help="--codec lzma2: 1 = price-based parse (stage C + stage P: what levels >= 5 / FLZMA2 >= 3 select in the codec module; the default), 0 = stage F + stage G's parse")
    ap.add_argument("--frame-log", type=int, default=0, help="log2 of the independent frame / block size (default: 20 for zstd; 23 = the 8 MiB dictionary of flzma2 -mx5 for --codec lzma2)")
    ap.add_argument("--lzma2-slice-log", type=int, default=-1, help="--codec lzma2: log2 of state-reset slices per block (default: the library's, 2)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--one-process", action="store_true",
                    help="no torchrun: ONE process, one context over --gpus N devices (b200z_create_multi), the whole --size-mib input through the host-pointer calls "
                         "(strong scaling: what one ICompressCoder::Code() call gets from the box)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned (compressed stream, decompressed "
                                                          "bytes) to DIR as .npy files, for comparing two builds output for output")
    return ap.parse_args()


# ---------------------------------------------------------------- clocks sampler (nvidia-smi)
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx = gpu_index; self.samples = []; self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True); self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for t, line in self.samples:
            if t < t0 or t > t1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1])); mx = float(f[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------- CPU reference arm
def cpu_reference(sample_bytes, seed_offset=0, level=3):
    """The reference's own CPU implementation of the path (oracle/_ref/libref_zstd.so compiled from
    /root/reference/C/zstd): the given level (3 = the headline), zstdmt with all host threads for encode (ZstdEncoder.cpp:300
    nbWorkers = #CPUs), single-threaded decode (ZstdDecoder.cpp:260-263: SetNumberOfThreads is a no-op)."""
    import ctypes
    import numpy as np
    import helpers
    import __graft_entry__ as ge
    pkg = ge.load_package()
    cores = os.cpu_count() or 1
    data = pkg.corpus.g2(sample_bytes, offset=seed_offset)
    if helpers.ref_available():
        Z = helpers.ref(); kind = "reference"
        out = np.zeros(Z.ZSTD_compressBound(sample_bytes), dtype=np.uint8)      # pre-faulted: page faults are not the codec
        c = Z.ZSTD_createCCtx()
        Z.ZSTD_CCtx_setParameter(c, 100, level); Z.ZSTD_CCtx_setParameter(c, 400, min(cores, 200))
        t = time.perf_counter(); r = Z.ZSTD_compress2(c, out.ctypes.data, out.size, data.ctypes.data, sample_bytes); t_enc = time.perf_counter() - t
        Z.ZSTD_freeCCtx(c)
        back = np.zeros(sample_bytes, dtype=np.uint8)
        t = time.perf_counter(); d = Z.ZSTD_decompress(back.ctypes.data, sample_bytes, out.ctypes.data, r); t_dec = time.perf_counter() - t
        assert d == sample_bytes
        enc_threads, dec_threads = min(cores, 200), 1
    else:                                                   # oracle port (single-threaded C restatement)
        O = helpers.oracle(); kind = "port"
        p = helpers.enc_params(**({"flags": 1 | 0x20} if level >= 8 else {}))
        out = np.empty(O.b2zo_zstd_compress_bound(sample_bytes, ctypes.byref(p)), dtype=np.uint8)
        t = time.perf_counter(); r = O.b2zo_zstd_compress(out.ctypes.data, out.size, data.ctypes.data, sample_bytes, ctypes.byref(p)); t_enc = time.perf_counter() - t
        back = np.empty(sample_bytes, dtype=np.uint8)
        t = time.perf_counter(); d = O.b2zo_zstd_decompress(back.ctypes.data, sample_bytes, out.ctypes.data, r); t_dec = time.perf_counter() - t
        assert d == sample_bytes
        enc_threads, dec_threads = 1, 1
    mb = sample_bytes / 1e6
    return {"value": mb / (t_enc + t_dec), "unit": "MB/s", "cores": cores, "kind": kind,
            "sample": f"{sample_bytes >> 20} MiB of the same G2 text, zstd level {level}: encode {enc_threads} threads (zstdmt), decode {dec_threads} thread (reference decoder is single-threaded)",
            "enc_MBps": mb / t_enc, "dec_MBps": mb / t_dec, "ratio": sample_bytes / r, "t_enc_s": t_enc, "t_dec_s": t_dec}


def cpu_reference_long(data, level, job_mib=0):
    """configs[2] on the host cores: the reference's encoder as `-m0=zstd:x<level>:long=27` sets it (ZstdEncoder.cpp:300-331: level,
    nbWorkers = #CPUs, enableLongDistanceMatching, windowLog 27) on `data` (a numpy sample of the G3 input).  job_mib != 0 sets
    ZSTD_c_jobSize: zstdmt's default job for a 128 MiB window is 512 MiB -- two jobs per GiB, two busy threads -- so the level-19
    sample is run with smaller jobs to use the cores within the bench's time; the ratio it gets is the reference's at that job size."""
    import numpy as np
    import helpers
    Z = helpers.ref()
    cores = os.cpu_count() or 1
    n = data.size
    c = Z.ZSTD_createCCtx()
    for k, v in ((100, level), (160, 1), (101, 27), (400, min(cores, 200))) + (((402, job_mib << 20),) if job_mib else ()):
        Z.ZSTD_CCtx_setParameter(c, k, v)
    out = np.zeros(Z.ZSTD_compressBound(n), dtype=np.uint8)
    t = time.perf_counter(); r = Z.ZSTD_compress2(c, out.ctypes.data, out.size, data.ctypes.data, n); t_enc = time.perf_counter() - t
    Z.ZSTD_freeCCtx(c)
    assert not Z.ZSTD_isError(r)
    back = np.zeros(n, dtype=np.uint8)
    t = time.perf_counter(); d = Z.ZSTD_decompress(back.ctypes.data, n, out.ctypes.data, r); t_dec = time.perf_counter() - t
    assert d == n
    mb = n / 1e6
    return {"value": mb / (t_enc + t_dec), "unit": "MB/s", "cores": cores, "kind": "reference", "level": level,
            "sample": f"first {n >> 20} MiB of the same G3 input, zstd level {level} long=27, {min(cores, 200)} workers, job size {str(job_mib) + ' MiB' if job_mib else 'default (4 windows)'}",
            "enc_MBps": mb / t_enc, "dec_MBps": mb / t_dec, "ratio": n / r}


def long_range(pkg, local, mib, cpu=True):
    """BASELINE configs[2]: text with long-range redundancy (G3: every 64 MiB a span of 1-4 MiB copied from up to 128 MiB back, 0.1 %
    of its bytes changed), `long=27`: the engine's long mode (frames of 1 GiB, window 128 MiB, stage L), resident in HBM, one timed
    pass after a warm-up; the plain mode on the same bytes beside it, and the reference's levels 3 and 19 with long=27 on a sample."""
    import torch
    n = mib << 20
    host = pkg.corpus.g3(n)
    d_in = torch.from_numpy(host).cuda()
    rec = {"workload": f"zstd long=27 (window 128 MiB, frames of 1 GiB), {mib} MiB G3 (G2 text + far copies, seed 3) resident in HBM, 1 timed pass"}
    for name, params in (("plain", {}), ("long27", {"long": 27})):
        c = pkg.Codec(local, **params)
        d_comp = torch.empty(c.compress_bound(n), dtype=torch.uint8, device="cuda"); d_back = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
        wn = n                                                              # warm-up at the full size: the scratch arenas grow here, not inside the timed pass
        m = c.compress_device(d_in.data_ptr(), wn, d_comp.data_ptr(), d_comp.numel()); c.decompress_device(d_comp.data_ptr(), m, d_back.data_ptr(), wn)
        c.reset_stats(); torch.cuda.synchronize()
        t0 = time.perf_counter(); m = c.compress_device(d_in.data_ptr(), n, d_comp.data_ptr(), d_comp.numel()); torch.cuda.synchronize(); t1 = time.perf_counter()
        r = c.decompress_device(d_comp.data_ptr(), m, d_back.data_ptr(), n); torch.cuda.synchronize(); t2 = time.perf_counter()
        assert r == n and torch.equal(d_back[:n], d_in), "long-range round trip mismatch"
        mb = n / 1e6
        rec[name] = {"value": mb / (t2 - t0), "unit": "MB/s", "enc_MBps": mb / (t1 - t0), "dec_MBps": mb / (t2 - t1), "ratio": n / m,
                     "kernel_ms": {k: c.stat(v) for k, v in dict(find_and_ldm=1, parse=10, entropy=2, assemble=3, dec_prepass=9, dec_entropy=4, dec_exec=5).items()}}
        c.close(); del d_comp, d_back
    rec["value"] = rec["long27"]["value"]; rec["unit"] = "MB/s"; rec["ratio"] = rec["long27"]["ratio"]
    rec["gain_over_plain_pct"] = 100.0 * (rec["long27"]["ratio"] / rec["plain"]["ratio"] - 1.0)
    del d_in
    torch.cuda.empty_cache()
    if cpu:
        import helpers
        if helpers.ref_available():
            sample = host[:min(n, 1 << 30)]
            c = pkg.Codec(local, long=27)                                  # the same sample through the engine, for a like-for-like ratio
            ours = len(c.compress(sample)); c.close()
            rec["sample_ratio"] = sample.size / ours
            cb = cpu_reference_long(sample, 3)
            cb["ratio_delta_pct"] = 100.0 * (rec["sample_ratio"] / cb["ratio"] - 1.0)
            rec["cpu_reference_L3"] = cb
            try:                                                           # level 19 takes minutes per GiB: measured once with tools/ref_cfg3.py on the same sample
                l19 = json.load(open(os.path.join(ROOT, "profiles", "r2_cfg3_reference.json")))["L19"]
                rec["reference_L19_recorded"] = {"ratio": l19["ratio"], "enc_MBps": l19["enc_MBps"], "cores": l19["cores"], "sample_MiB": l19["sample_MiB"], "job_MiB": l19["jobSize_MiB"],
                                                 "ratio_delta_pct": 100.0 * (rec["sample_ratio"] / l19["ratio"] - 1.0), "source": "profiles/r2_cfg3_reference.json"}
            except Exception:
                pass
    return rec


def reference_streams(pkg, local, mib=1024, lz_mib=64):
    """Streams the REFERENCE wrote, through the engine's host-pointer decoders (what the codec module's CDecoder does with a stock archive):
    zstd level 3 from zstdmt -- ONE frame whatever the thread count (jobs become blocks of one frame, zstdmt_compress.c:1403), 2 MiB sliding
    window -- and the stock LZMA2 encoder at level 5 (`-m0=lzma2 -mx5`: Lzma2Enc.c, 16 MiB dictionary, a dictionary reset per 64 MiB block
    when it runs block-threaded).  The zstd frame's blocks are entropy-decoded in parallel and its matches resolved by pointer jumping
    (stage J, csrc/zstd_dec.cu; `units_ms`: the same stream through the execution units, which form one chain on it); the same frame with a
    content checksum -- what the reference's .zst handler writes (ZstdHandler.cpp:262-282) -- adds one XXH64 over the whole output, four
    sequential accumulators whatever the machine; a raw LZMA2 stream is one chain per dictionary reset."""
    import numpy as np, torch
    import helpers
    rec = {}
    if not helpers.ref_available():
        return {"unavailable": "oracle/_ref/libref_zstd.so missing"}
    cores = os.cpu_count() or 1
    n = mib << 20
    data = pkg.corpus.g2(n)
    c = pkg.Codec(local)
    comp = helpers.ref_compress(data, level=3, nbWorkers=min(cores, 64))
    hc = torch.from_numpy(np.frombuffer(comp, dtype=np.uint8).copy()).pin_memory(); hb = torch.empty(n, dtype=torch.uint8).pin_memory()
    c.decompress_into(hc.data_ptr(), len(comp), hb.data_ptr(), n)                      # warm-up (allocations)
    c.reset_stats()
    t = time.perf_counter(); r = c.decompress_into(hc.data_ptr(), len(comp), hb.data_ptr(), n); dt = time.perf_counter() - t
    assert r == n and torch.equal(hb, torch.from_numpy(data)), "reference-written zstd stream: round trip mismatch"
    rec["zstd_single_frame"] = {"workload": f"{mib} MiB G2 text, reference zstd level 3 ({min(cores, 64)} workers): one frame, window 2 MiB", "packed_bytes": len(comp),
                                "dec_MBps": n / 1e6 / dt, "ms": dt * 1e3, "frames_by_pointer_jumping": int(c.stat(11)),
                                "kernel_ms": {k: c.stat(v) for k, v in dict(prepass=9, entropy=4, layout_exec_verify=5).items()}}
    # the same frame with a content checksum (one XXH64 chain over the output), and through the execution units on a quarter of it
    comp_ck = helpers.ref_compress(data, level=3, checksum=1, nbWorkers=min(cores, 64))
    hk = torch.from_numpy(np.frombuffer(comp_ck, dtype=np.uint8).copy()).pin_memory()
    c.reset_stats()
    t = time.perf_counter(); r = c.decompress_into(hk.data_ptr(), len(comp_ck), hb.data_ptr(), n); dt = time.perf_counter() - t
    assert r == n and torch.equal(hb, torch.from_numpy(data)), "reference-written zstd stream with checksum: round trip mismatch"
    rec["zstd_single_frame"]["with_content_checksum"] = {"dec_MBps": n / 1e6 / dt, "ms": dt * 1e3, "layout_exec_verify_ms": c.stat(5)}
    q = n >> 2
    comp_q = helpers.ref_compress(data[:q], level=3, nbWorkers=min(cores, 64))
    hq = torch.from_numpy(np.frombuffer(comp_q, dtype=np.uint8).copy()).pin_memory()
    cu = pkg.Codec(local, dec_jump=0)
    t = time.perf_counter(); r = cu.decompress_into(hq.data_ptr(), len(comp_q), hb.data_ptr(), q); dtu = time.perf_counter() - t
    assert r == q
    cu.close()
    rec["zstd_single_frame"]["units_ms"] = {"sample_MiB": q >> 20, "ms": dtu * 1e3, "dec_MBps": q / 1e6 / dtu}
    del hc, hb, hk, hq
    if helpers.ref_lzma_available():
        m = lz_mib << 20
        prop, lcomp = helpers.ref_lzma2_compress(data[:m], 5, threads=min(cores, 32))
        blocks = c.lzma2_stream_info(lcomp)[1]
        hc = torch.from_numpy(np.frombuffer(lcomp, dtype=np.uint8).copy()).pin_memory(); hb = torch.empty(m, dtype=torch.uint8).pin_memory()
        wprop, wcomp = helpers.ref_lzma2_compress(data[:1 << 20], 5)                    # warm-up on a small stream (one chain of 64 MiB takes seconds)
        wc = torch.from_numpy(np.frombuffer(wcomp, dtype=np.uint8).copy()).pin_memory()
        c.lzma2_decompress_into(wc.data_ptr(), len(wcomp), wprop, hb.data_ptr(), 1 << 20)
        t = time.perf_counter(); r = c.lzma2_decompress_into(hc.data_ptr(), len(lcomp), prop, hb.data_ptr(), m); dt = time.perf_counter() - t
        assert r == m and torch.equal(hb, torch.from_numpy(data[:m])), "reference-written LZMA2 stream: round trip mismatch"
        rec["lzma2_mx5"] = {"workload": f"{lz_mib} MiB G2 text, reference Lzma2Enc level 5 ({min(cores, 32)} threads)", "packed_bytes": len(lcomp), "independent_blocks": int(blocks),
                            "dec_MBps": m / 1e6 / dt, "ms": dt * 1e3}
    c.close()
    return rec


def cpu_reference_lzma2(sample_bytes, seed_offset=0):
    """Method 21 on the host cores, the way the reference's coders run it: Fast-LZMA2 level 5 with all threads for encode
    (CFastEncoder -> FL2_compressStream, Lzma2Encoder.cpp:280-340; FL2_compressMt keeps the same level table and reset
    interval) and the multi-threaded LZMA2 decoder for decode (Lzma2Decoder.cpp:95-186 -> Lzma2DecMt_Decode, driven by
    oracle/ref_harness/lzma2_decmt_harness.c with memory streams)."""
    import helpers
    import __graft_entry__ as ge
    pkg = ge.load_package()
    cores = os.cpu_count() or 1
    if not helpers.ref_lzma_available():
        raise SystemExit("bench.py --codec lzma2: oracle/_ref/libref_lzma.so missing (built by __graft_entry__.build() where /root/reference exists)")
    data = pkg.corpus.g2(sample_bytes, offset=seed_offset).tobytes()
    t = time.perf_counter(); prop, comp = helpers.ref_fl2_compress(data, 5, threads=0); t_enc = time.perf_counter() - t
    t = time.perf_counter(); back, mt = helpers.ref_lzma2_decompress_mt(comp, sample_bytes, prop, min(cores, 64)); t_dec = time.perf_counter() - t
    assert back == data
    mb = sample_bytes / 1e6
    return {"value": mb / (t_enc + t_dec), "unit": "MB/s", "cores": cores, "kind": "reference",
            "sample": f"{sample_bytes >> 20} MiB of the same G2 text: Fast-LZMA2 level 5 encode on all threads (FL2_compressMt), reference MT decoder "
                      f"({min(cores, 64)} threads; ran {'multi' if mt else 'single'}-threaded: parallelism = dictionary resets in the stream)",
            "enc_MBps": mb / t_enc, "dec_MBps": mb / t_dec, "ratio": sample_bytes / len(comp), "t_enc_s": t_enc, "t_dec_s": t_dec}


def one_call_multi_gpu(pkg, devices, host_in, unit_bytes, steps, lz=False):
    """one context over `devices`: the host-pointer compress + decompress of the SAME input (strong scaling), pinned host buffers"""
    import torch
    c = pkg.Codec(devices=devices)
    bound = c.compress_bound(unit_bytes)
    host_comp = torch.empty(bound, dtype=torch.uint8).pin_memory()
    host_back = torch.empty(unit_bytes, dtype=torch.uint8).pin_memory()
    n = c.compress_into(host_in.data_ptr(), unit_bytes, host_comp.data_ptr(), bound)          # warm-up (allocations, first touches)
    c.decompress_into(host_comp.data_ptr(), n, host_back.data_ptr(), unit_bytes)
    t_enc = t_dec = 0.0
    for _ in range(steps):
        t0 = time.perf_counter(); n = c.compress_into(host_in.data_ptr(), unit_bytes, host_comp.data_ptr(), bound); t1 = time.perf_counter()
        m = c.decompress_into(host_comp.data_ptr(), n, host_back.data_ptr(), unit_bytes); t2 = time.perf_counter()
        assert m == unit_bytes
        t_enc += t1 - t0; t_dec += t2 - t1
    assert torch.equal(host_back, host_in)
    c.close()
    mb = steps * unit_bytes / 1e6
    return {"devices": len(devices), "uncompressed_bytes": unit_bytes, "value": mb / (t_enc + t_dec), "unit": "MB/s", "enc_MBps": mb / t_enc, "dec_MBps": mb / t_dec,
            "ratio": unit_bytes / n, "what": "ONE process, ONE context over all devices, one compress_host + decompress_host call per step on the same input (strong scaling)"}


def many_files_7z(pkg, codec, n_files=100_000, file_bytes=65536, cpu_files=4000, cpu=True):
    """BASELINE configs[4]: n_files mixed-entropy files (SURVEY.md 8(d) cfg5 classes: half text, noise, 16-symbol skew, tiled) -> ONE
    b200z_7z_write_archive_host call (non-solid: one folder per file).  Beside it the reference's `7zz a -m0=zstd -mx3 -ms=off` on a bounded
    sample of the same files from tmpfs, all host threads."""
    import numpy as np, tempfile, shutil
    text = pkg.corpus.g2(n_files * file_bytes // 2)
    buf = np.concatenate([text, pkg.corpus.entropy_class(1, n_files * file_bytes // 8), pkg.corpus.entropy_class(2, n_files * file_bytes // 8),
                          pkg.corpus.entropy_class(3, n_files * file_bytes // 4)])[: n_files * file_bytes]
    order = np.random.RandomState(5).permutation(n_files)                     # interleave the classes
    buf = np.ascontiguousarray(buf.reshape(n_files, file_bytes)[order]).reshape(-1)
    import torch, ctypes
    hin = torch.from_numpy(buf).pin_memory()
    sizes = np.full(n_files, file_bytes, dtype=np.uint64)
    names = [f"d{i % 100:02d}/f{i:06d}.bin".encode() for i in range(n_files)]
    arr = (ctypes.c_char_p * n_files)(*names)
    cap = codec.L.b200z_7z_archive_bound(codec.h, buf.nbytes, n_files, sum(len(x) + 1 for x in names))
    hout = torch.empty(cap, dtype=torch.uint8).pin_memory(); n = ctypes.c_size_t()
    best = None
    for _ in range(2):                                                         # first call: allocations
        t = time.perf_counter()
        rc = codec.L.b200z_7z_write_archive_host(codec.h, hin.data_ptr(), sizes.ctypes.data, arr, None, n_files, hout.data_ptr(), cap, ctypes.byref(n))
        t = time.perf_counter() - t
        assert rc == 0, codec.L.b200z_last_error(codec.h)
        best = t
    rec = {"workload": f"{n_files} files x {file_bytes} B (text / noise / skew / tiles), one non-solid .7z (method ZSTD level 3, one folder per file), pinned host buffers, one call",
           "value": buf.nbytes / 1e6 / best, "unit": "MB/s", "files_per_s": n_files / best, "ms": 1e3 * best, "ratio": buf.nbytes / n.value, "archive_bytes": n.value}
    stock = os.path.join(ROOT, "oracle", "_ref", "7z", "stock", "7zz")
    if cpu and os.path.exists(stock):
        d = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            # the archive just written, tested by the reference itself (a sample archive of the first files: the stock decoder is single-threaded)
            k = min(cpu_files, n_files)
            for i in range(k):
                os.makedirs(os.path.join(d, "in", f"d{i % 100:02d}"), exist_ok=True)
                buf[i * file_bytes:(i + 1) * file_bytes].tofile(os.path.join(d, "in", names[i].decode()))
            cores = os.cpu_count() or 1
            t = time.perf_counter()
            r = subprocess.run([stock, "a", "-m0=zstd", "-mx3", "-ms=off", f"-mmt={cores}", "-bso0", "-bsp0", os.path.join(d, "ref.7z"), "."], cwd=os.path.join(d, "in"), capture_output=True, text=True)
            t = time.perf_counter() - t
            if r.returncode == 0:
                rec["cpu_baseline"] = {"value": k * file_bytes / 1e6 / t, "unit": "MB/s", "files_per_s": k / t, "cores": cores, "kind": "reference",
                                       "sample": f"7zz a -m0=zstd -mx3 -ms=off -mmt={cores} on the first {k} of the same files from tmpfs",
                                       "ratio": k * file_bytes / os.path.getsize(os.path.join(d, "ref.7z"))}
            ours = codec.write_7z([buf[i * file_bytes:(i + 1) * file_bytes].tobytes() for i in range(k)], [x.decode() for x in names[:k]])
            open(os.path.join(d, "ours.7z"), "wb").write(ours)
            r = subprocess.run([stock, "t", os.path.join(d, "ours.7z")], capture_output=True, text=True)
            rec["reference_7zz_verifies_sample_archive"] = bool(r.returncode == 0 and "Everything is Ok" in r.stdout)
        finally:
            shutil.rmtree(d, ignore_errors=True)
    return rec


def dump_outputs(out_dir, d_comp, csize, d_back, prop=None, sample=4 << 20, chunk=1 << 20):
    """What one step of the timed path returned, as float32 / float64 .npy files in out_dir (32 MB for the default 4 GiB):
    compressed_size (and lzma2_prop), a seeded sample of `sample` bytes of the compressed stream and of the decompressed output
    (the same positions in every run with the same arguments), and the sum of every `chunk` bytes of both, so that a difference
    anywhere shows."""
    import numpy as np, torch
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "compressed_size.npy"), np.array([csize], dtype=np.float64))
    if prop is not None:
        np.save(os.path.join(out_dir, "lzma2_prop.npy"), np.array([prop], dtype=np.float64))
    for name, t in (("compressed", d_comp[:csize]), ("decompressed", d_back)):
        n = t.numel()
        idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, sample), replace=False))
        np.save(os.path.join(out_dir, f"{name}_sample.npy"), t[torch.from_numpy(idx).to(t.device)].cpu().numpy().astype(np.float32))
        sums = torch.stack([t[i:i + chunk].sum(dtype=torch.int64) for i in range(0, n, chunk)]) if n else torch.zeros(0, dtype=torch.int64)
        np.save(os.path.join(out_dir, f"{name}_chunk_sums.npy"), sums.cpu().numpy().astype(np.float64))


def bind_to_gpu_numa_node(index):
    """Run this rank on the cores of the NUMA node its GPU hangs off, BEFORE any pinned buffer is allocated (first touch then places the
    staging memory next to the GPU's PCIe root: 8 ranks x 12 GB of H2D + D2H per step otherwise cross the socket link for half the GPUs).
    Best effort: returns the node or None and never raises."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]                                               # nvml prints an 8-digit PCI domain, sysfs a 4-digit one
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        cpus = set()
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def main():
    a = parse_args()
    lz = a.codec == "lzma2"
    cpu_ref = cpu_reference_lzma2 if lz else (lambda nbytes, seed_offset=0: cpu_reference(nbytes, seed_offset, a.level))
    metric_name = "LZMA2 (method 21) encode+decode throughput" if lz else f"zstd-L{a.level} encode+decode throughput"
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    unit_bytes = a.size_mib << 20
    workload = f"zstd level {a.level}, {a.size_mib} MiB synthetic enwik-shape text (generator G2) per GPU, 128 KiB blocks"
    if lz:
        workload = f"LZMA2 / Fast-LZMA2 coder (method 21), {a.size_mib} MiB synthetic enwik-shape text (generator G2) per GPU, {1 << ((a.frame_log or 23) - 20)} MiB dictionary-reset blocks, parse {a.lzma2_parse}"

    if a.impl == "reference":
        if rank != 0:
            return
        sample = a.cpu_sample_mib << 20
        for _ in range(max(0, min(a.warmup, 1))):
            cpu_ref(min(sample, 64 << 20))
        t_tot = 0.0; res = None
        for _ in range(a.steps):
            res = cpu_ref(sample); t_tot += res["t_enc_s"] + res["t_dec_s"]
        value = a.steps * sample / 1e6 / t_tot
        line = {"impl": "reference", "metric": metric_name, "value": value, "unit": "MB/s", "n_gpus": a.gpus,
                "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * t_tot / a.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": workload, "sample": res["sample"]},
                "cpu_baseline": {k: res[k] for k in ("unit", "cores", "kind", "sample", "enc_MBps", "dec_MBps", "ratio")} | {"value": value},
                "e2e": {"value": value, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line)); return

    import numpy as np
    import torch
    import __graft_entry__ as ge
    pkg = ge.load_package()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU fallback)")
    if a.one_process:
        if lz:
            raise SystemExit("--one-process: the multi-device dispatcher serves the zstd host calls")
        ndev = min(a.gpus, torch.cuda.device_count())
        host_in = torch.empty(unit_bytes, dtype=torch.uint8).pin_memory()
        pkg.corpus.g2_into(host_in.data_ptr(), unit_bytes)
        res = one_call_multi_gpu(pkg, list(range(ndev)), host_in, unit_bytes, a.steps)
        print(json.dumps({"metric": metric_name + " (one call, all devices)", "value": res["value"], "unit": "MB/s", "n_gpus": ndev, "steps": a.steps, "warmup": 1,
                          "higher_is_better": True, "scaling": "strong", "dtype": "u8", "data": "synthetic", "config": {"workload": workload.replace(" per GPU", " in total")}, "e2e": res}))
        return
    torch.cuda.set_device(local)
    numa_node = bind_to_gpu_numa_node(local) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        cpu_group = dist.new_group(backend="gloo")                      # for waits that must leave the GPUs idle (an NCCL barrier spins on the device)

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    codec = pkg.Codec(local)
    if lz and not a.frame_log:
        a.frame_log = 23                                            # fl2_compress.c:80: level 5 = 8 MiB dictionary; a frame = one dictionary-reset block
    if a.frame_log:
        codec.set("frame_log", a.frame_log); codec.set("window_log", a.frame_log)
    if not lz and a.level != 3:
        codec.set("level", a.level)
    if lz and a.lzma2_slice_log >= 0:
        codec.set("lzma2_slice_log", a.lzma2_slice_log)
    if lz and a.lzma2_parse:
        codec.set("lzma2_parse", 1)
    # ---- corpus shard: rank r owns bytes [r*unit, (r+1)*unit) of the seeded G2 stream (weak scaling)
    host_in = torch.empty(unit_bytes, dtype=torch.uint8).pin_memory()
    pkg.corpus.g2_into(host_in.data_ptr(), unit_bytes, offset=rank * unit_bytes, threads=max(1, (os.cpu_count() or 8) // max(1, world)))
    d_in = host_in.cuda(non_blocking=False)
    bound = codec.lzma2_compress_bound(unit_bytes) if lz else codec.compress_bound(unit_bytes)
    d_comp = torch.empty(bound, dtype=torch.uint8, device="cuda")
    d_back = torch.empty(unit_bytes, dtype=torch.uint8, device="cuda")

    last = {}

    def step_device():
        if lz:
            t0 = time.perf_counter(); c, prop = codec.lzma2_compress_device(d_in.data_ptr(), unit_bytes, d_comp.data_ptr(), bound); t1 = time.perf_counter()
            n = codec.lzma2_decompress_device(d_comp.data_ptr(), c, prop, d_back.data_ptr(), unit_bytes); t2 = time.perf_counter()
            assert n == unit_bytes
            last["prop"] = prop
            return c, t1 - t0, t2 - t1
        t0 = time.perf_counter(); c = codec.compress_device(d_in.data_ptr(), unit_bytes, d_comp.data_ptr(), bound); t1 = time.perf_counter()
        n = codec.decompress_device(d_comp.data_ptr(), c, d_back.data_ptr(), unit_bytes); t2 = time.perf_counter()
        assert n == unit_bytes
        return c, t1 - t0, t2 - t1

    for _ in range(a.warmup):
        csize, _, _ = step_device()
    assert torch.equal(d_back, d_in), "round trip mismatch"                      # bit-exact round trip (outside the timed region)
    ratio = unit_bytes / csize

    sampler = ClockSampler(local); sampler.start()
    codec.reset_stats()
    barrier(); T0 = time.perf_counter()
    t_enc = t_dec = 0.0
    for _ in range(a.steps):
        csize, te, td = step_device(); t_enc += te; t_dec += td
    barrier(); T1 = time.perf_counter()
    clocks = sampler.stop(T0, T1)
    elapsed = T1 - T0
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, d_comp, csize, d_back, last.get("prop"))
    stats = {k: codec.stat(v) for k, v in dict(match_ms=1, entropy_ms=2, assemble_ms=3, dec_prepass_ms=9, dec_entropy_ms=4, dec_exec_ms=5, launches=6, parse_ms=10).items()}
    if dist:
        t = torch.tensor([elapsed, t_enc, t_dec], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX); elapsed, t_enc, t_dec = (float(x) for x in t.cpu())
    units_mb = world * a.steps * unit_bytes / 1e6
    value = units_mb / elapsed

    # ---- end to end through the host-pointer C ABI (what the 7-Zip coder wrapper calls): pinned host
    #      buffers, H2D of the input and D2H of the result inside the timed region
    e2e = None
    if not a.no_e2e:
        host_comp = torch.empty(bound, dtype=torch.uint8).pin_memory()
        host_back = torch.empty(unit_bytes, dtype=torch.uint8).pin_memory()

        def step_host():
            if lz:
                c, prop = codec.lzma2_compress_into(host_in.data_ptr(), unit_bytes, host_comp.data_ptr(), bound)
                n = codec.lzma2_decompress_into(host_comp.data_ptr(), c, prop, host_back.data_ptr(), unit_bytes)
                assert n == unit_bytes
                return c
            c = codec.compress_into(host_in.data_ptr(), unit_bytes, host_comp.data_ptr(), bound)
            n = codec.decompress_into(host_comp.data_ptr(), c, host_back.data_ptr(), unit_bytes)
            assert n == unit_bytes
            return c
        c = step_host()
        barrier(); E0 = time.perf_counter()
        for _ in range(a.steps):
            c = step_host()
        barrier(); E1 = time.perf_counter()
        assert torch.equal(host_back, host_in)
        e_el = E1 - E0
        if dist:
            t = torch.tensor([e_el], device="cuda", dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); e_el = float(t.cpu()[0])
        e2e = {"value": units_mb / e_el, "unit": "MB/s", "h2d_bytes_per_step": world * (unit_bytes + c), "d2h_bytes_per_step": world * (c + unit_bytes)}

    # ---- one call on all N devices (rank 0; the other ranks wait): the dispatcher inside the product, strong scaling on ONE rank's input
    multi = None
    if dist and not lz and not a.no_e2e:
        barrier()
        if rank != 0:
            codec.close(); del d_in, d_comp, d_back; torch.cuda.empty_cache()      # the other ranks leave their GPUs to rank 0's context ...
        if rank == 0:
            try:
                multi = one_call_multi_gpu(pkg, list(range(world)), host_in, unit_bytes, max(1, min(a.steps, 3)))
            except Exception as e:                                   # e.g. ranks not on devices 0..N-1 of this process's view
                multi = {"error": str(e)[:200]}
        dist.barrier(group=cpu_group)                                # ... and wait on the CPU
    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel (stage F, zstd_enc_find_kernel): algorithmic bytes per launch
    #      = U * (1 + 1/ratio)  (SURVEY.md 8(d): encode reads the input once, writes the compressed stream once)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0); peak_src = "measured" if "hbm_gbs" in peaks else "fallback"
    # LZMA2: the dominant kernel is stage R (lzma2_enc_range_kernel: one serial range-coder chain per 1 MiB block)
    #        with the price-based parse it is stage P (lzma2_parse_kernel: one dynamic-programme chain per slice)
    zparse = (not lz) and a.level >= 8
    dom_kernel = ("lzma2_parse_kernel" if a.lzma2_parse else "lzma2_enc_range_kernel") if lz else ("zstd_enc_parse_kernel" if zparse else "zstd_enc_find_kernel")
    match_ms = ((stats["parse_ms"] if a.lzma2_parse else stats["entropy_ms"]) if lz else (stats["parse_ms"] if zparse else stats["match_ms"])) / a.steps
    algo_bytes = unit_bytes * (1.0 + 1.0 / ratio)
    achieved = algo_bytes / 1e9 / (match_ms / 1e3) if match_ms > 0 else 0.0
    traffic = None
    try:
        if not (lz and a.lzma2_parse) and not zparse:               # no ncu capture of stage P / stage Z yet
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r1_lzma2_range_traffic.json" if lz else "r2_find_traffic.json")))["dram_bytes_per_input_byte"] * unit_bytes
    except Exception:
        pass
    line = {
        "metric": metric_name, "value": value, "unit": "MB/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * elapsed / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload, "global_uncompressed_bytes_per_step": world * unit_bytes, "frame_log": codec.get("frame_log"),
                   "parallelism": f"{world} independent shard(s), no collective", **({"lzma2_parse": a.lzma2_parse} if lz else {"level": a.level}), "l2": f"inputs ({a.size_mib} MiB per GPU) larger than L2; no flush needed",
                   "host_batch_log": codec.get("host_batch_log"), "rank0_numa_node": numa_node,
                   "ratio": ratio, "enc_MBps": units_mb / t_enc, "dec_MBps": units_mb / t_dec,
                   "kernel_ms_per_step": {k: v / a.steps for k, v in stats.items() if k != "launches"}},
        "roofline": {"bound": "hbm", "kernel": dom_kernel, "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": match_ms},
        "clocks": clocks, "gpu_launches": int(stats["launches"]), "e2e": e2e,
    }
    if multi:
        line["extra"] = {"one_call_multi_gpu": multi}
    if not lz and world == 1 and not a.no_lzma2_extra:
        # BASELINE configs[3] beside the headline: method 21 the way `-m0=flzma2 -mx5` runs it in the codec module (price-based parse,
        # 8 MiB dictionary-reset blocks), the same 4 GiB resident in HBM, one timed pass after a small warm-up; the reference's FL2 level 5
        # on a bounded sample of the same text beside it
        del d_comp, d_back
        torch.cuda.empty_cache()
        lc = pkg.Codec(local, lzma2_parse=1, frame_log=23, window_log=23)
        lb = lc.lzma2_compress_bound(unit_bytes)
        l_comp = torch.empty(lb, dtype=torch.uint8, device="cuda"); l_back = torch.empty(unit_bytes, dtype=torch.uint8, device="cuda")
        wn = min(unit_bytes, 256 << 20)
        c0, p0 = lc.lzma2_compress_device(d_in.data_ptr(), wn, l_comp.data_ptr(), lb); lc.lzma2_decompress_device(l_comp.data_ptr(), c0, p0, l_back.data_ptr(), wn)
        lc.reset_stats(); torch.cuda.synchronize()
        t0 = time.perf_counter(); c1, p1 = lc.lzma2_compress_device(d_in.data_ptr(), unit_bytes, l_comp.data_ptr(), lb); t1 = time.perf_counter()
        nb = lc.lzma2_decompress_device(l_comp.data_ptr(), c1, p1, l_back.data_ptr(), unit_bytes); t2 = time.perf_counter()
        assert nb == unit_bytes and torch.equal(l_back, d_in), "LZMA2 round trip mismatch"
        mbs = unit_bytes / 1e6
        lz_rec = {"workload": f"method 21, price-based parse, 8 MiB dictionary-reset blocks, {a.size_mib} MiB G2 text resident in HBM, 1 pass", "value": mbs / (t2 - t0), "unit": "MB/s",
                  "enc_MBps": mbs / (t1 - t0), "dec_MBps": mbs / (t2 - t1), "ratio": unit_bytes / c1,
                  "kernel_ms": {k: lc.stat(v) for k, v in dict(stage_c=1, stage_p=10, stage_r=2, assemble=3, dec_prepass=9, dec=4).items()}}
        if not a.no_cpu_baseline:
            try:
                cb2 = cpu_reference_lzma2(min(unit_bytes, 512 << 20))
                lz_rec["cpu_baseline"] = {k: cb2[k] for k in ("value", "unit", "cores", "kind", "sample", "enc_MBps", "dec_MBps", "ratio")}
                lz_rec["ratio_delta_vs_reference_pct"] = 100.0 * (lz_rec["ratio"] / cb2["ratio"] - 1.0)
            except SystemExit as e:
                lz_rec["cpu_baseline"] = {"unavailable": str(e)[:120]}
        line.setdefault("extra", {})["lzma2"] = lz_rec
        lc.close()
        del l_comp, l_back
        torch.cuda.empty_cache()
    if not lz and world == 1 and not a.no_files_extra:
        try:
            line.setdefault("extra", {})["many_files_7z"] = many_files_7z(pkg, codec, cpu=not a.no_cpu_baseline)
        except Exception as e:
            line.setdefault("extra", {})["many_files_7z"] = {"error": str(e)[:200]}
    if not lz and world == 1 and not a.no_long_extra:
        try:
            del d_in
            torch.cuda.empty_cache()
            line.setdefault("extra", {})["long_range"] = long_range(pkg, local, a.long_mib, cpu=not a.no_cpu_baseline)
        except Exception as e:
            line.setdefault("extra", {})["long_range"] = {"error": str(e)[:200]}
    if not lz and world == 1 and not a.no_refstreams_extra and not a.no_cpu_baseline:
        try:
            line.setdefault("extra", {})["reference_streams"] = reference_streams(pkg, local)
        except Exception as e:
            line.setdefault("extra", {})["reference_streams"] = {"error": str(e)[:200]}
    if not a.no_cpu_baseline and world == 1:
        cb = cpu_ref(a.cpu_sample_mib << 20)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "enc_MBps", "dec_MBps", "ratio")}
    print(json.dumps(line))
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
