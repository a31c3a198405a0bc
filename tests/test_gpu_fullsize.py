"""Parity at BASELINE.json's full sizes and for the mixed stream (configs[2], [3], [4]), the independent Python
timestamp oracle, and the concurrency contract of decoder clones.  GPU only; every decode goes through the C ABI."""
import datetime
import os
import struct
import threading

import numpy as np
import pytest

from conftest import assert_parity

pytestmark = pytest.mark.gpu
NT = min(os.cpu_count() or 8, 32)


def _fullsize(native, oracle, fmt, seed, mean, total, sub, cfg=None, **kw):
    """`total` lines fed as int32-offset sub-batches of `sub` lines (how bench.py feeds configs[2]/[3]); every Record of
    every sub-batch is compared with the oracle."""
    dec = None
    done = 0
    try:
        while done < total:
            k = min(sub, total - done)
            data, offs = native.generate(fmt, seed, k, first_index=done, mean_len=mean, bad_frac=0.005, nthreads=NT)
            if dec is None:
                dec = native.BatchDecoder(fmt, max_batch_bytes=int(offs[-1]) + (64 << 20), max_batch_lines=sub, **kw)
            res = dec.decode(data, offs)
            step = 500_000  # bounds the dump buffers
            for lo in range(0, k, step):
                hi = min(k, lo + step)
                gbuf, goffs = dec.dump(res, data, offs, nthreads=NT, lo=lo, hi=hi)
                base = int(offs[lo])
                so = (offs[lo:hi + 1] - base).astype(np.int32)
                obuf, ooffs = oracle.decode_dump(fmt, data[base:int(offs[hi])], so, cfg, nthreads=NT)
                assert gbuf == obuf and np.array_equal(goffs, ooffs), f"lines {done + lo}:{done + hi} differ from the oracle"
            done += k
    finally:
        if dec is not None:
            dec.close()


def test_ltsv_10m_lines(native, oracle):
    """BASELINE.json configs[3]: 10 M LTSV lines (20 key:value fields), 2.5 M-line sub-batches."""
    _fullsize(native, oracle, native.FMT_LTSV, 1757, 420.0, 10_000_000, 2_500_000)


def test_gelf_10m_lines(native, oracle):
    """BASELINE.json configs[2]: 10 M GELF lines (mean 512 B), 2.5 M-line sub-batches."""
    _fullsize(native, oracle, native.FMT_GELF, 0x6E1F, 466.0, 10_000_000, 2_500_000)


def test_mixed_stream_c5_demux(native, oracle):
    """BASELINE.json configs[4] (one GPU's shard, reduced to 1.6 M lines): RFC5424 and GELF runs of 4096 lines
    interleaved; the host demultiplexes the runs into one batch per format exactly like bench.py::run_mixed, decodes each
    on its own Decoder, and every Record of the re-interleaved stream is compared with the oracle."""
    RUN, runs = 4096, 392
    parts = {0: [], 2: []}
    order = []
    idx = {0: 0, 2: 0}
    for r in range(runs):
        fmt = 0 if r % 2 == 0 else 2
        data, offs = native.generate(fmt, 5424 if fmt == 0 else 0x6E1F, RUN, first_index=idx[fmt],
                                     mean_len=169.2 if fmt == 0 else 466.0, bad_frac=0.005, nthreads=8)
        idx[fmt] += RUN
        parts[fmt].append((data, offs))
        order.append(fmt)
    for fmt in (0, 2):
        datas = [d for d, _ in parts[fmt]]
        lens = np.concatenate([np.diff(o) for _, o in parts[fmt]])
        offs = np.zeros(len(lens) + 1, dtype=np.int32)
        np.cumsum(lens, out=offs[1:])
        data = np.concatenate(datas)
        dec = native.BatchDecoder(fmt, max_batch_bytes=int(offs[-1]) + (1 << 20), max_batch_lines=len(lens))
        try:
            assert_parity(dec, oracle, fmt, data, offs)
            assert_parity(dec, oracle, fmt, data, offs, resident=True)  # what run_mixed times
        finally:
            dec.close()


def test_multi_device_fanout(native, oracle):
    """MultiGpuBatchDecoder on two REAL devices (skipped on a machine with fewer): byte-balanced shards, one context + host
    thread per device, Records gathered in order."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    for fmt, seed in ((native.FMT_RFC5424, 77), (native.FMT_GELF, 78), (native.FMT_LTSV, 79)):
        data, offs = native.generate(fmt, seed, 300_000)
        gbuf, goffs = native.multi_gpu_decode_dump(fmt, [0, 1], data, offs)
        obuf, ooffs = oracle.decode_dump(fmt, data, offs, None, nthreads=NT)
        assert gbuf == obuf and np.array_equal(goffs, ooffs)


def _py_rfc3339_ts(s: str) -> float:
    """Independent of the C++ oracle: datetime + integer arithmetic, then the reference's f64 recipe
    (utils/mod.rs:24-28): float(nanos_i128) / 1e9 — Python ints are exact, int -> float and / are IEEE round-to-nearest."""
    date, rest = s.split("T")
    y, mo, d = (int(x) for x in date.split("-"))
    if rest.endswith("Z"):
        off, core = 0, rest[:-1]
    else:
        sign = 1 if rest[-6] == "+" else -1
        off = sign * (int(rest[-5:-3]) * 3600 + int(rest[-2:]) * 60)
        core = rest[:-6]
    hms, _, frac = core.partition(".")
    h, mi, sec = (int(x) for x in hms.split(":"))
    nanos = int((frac + "000000000")[:9]) if frac else 0
    days = (datetime.date(y, mo, d) - datetime.date(1970, 1, 1)).days
    total = (days * 86400 + h * 3600 + mi * 60 + sec - off) * 1_000_000_000 + nanos
    return float(total) / 1e9


def test_timestamp_bits_vs_python_mini_oracle(native):
    """1 M generated RFC5424 stamps: the GPU's f64 bits equal float(nanos)/1e9 computed by Python (three-way check:
    C++ oracle <-> Python <-> GPU; the oracle side is covered by the dump comparisons)."""
    n = 1_000_000
    data, offs = native.generate(native.FMT_RFC5424, 31337, n, bad_frac=0.0)
    dec = native.BatchDecoder(native.FMT_RFC5424, max_batch_bytes=int(offs[-1]) + (1 << 20), max_batch_lines=n)
    try:
        res = dec.decode(data, offs)
        status = np.array(res.status)               # the result arrays belong to the context: copy before closing it
        got = np.array(res.ts).view(np.uint64)
    finally:
        dec.close()
    assert (status == 0).all()
    raw = data.tobytes()
    bad = 0
    for i in range(n):
        a = raw.index(b" ", int(offs[i])) + 1
        b = raw.index(b" ", a)
        want = struct.unpack("<Q", struct.pack("<d", _py_rfc3339_ts(raw[a:b].decode())))[0]
        if want != int(got[i]):
            bad += 1
            assert bad < 5, (raw[a:b], hex(want), hex(int(got[i])))
    assert bad == 0


def test_decoder_clones_decode_concurrently(native, oracle):
    """ADVICE r1: clones made by clone_boxed() share one context; concurrent decode() calls must serialise instead of
    racing on the context's buffers (two threads, 2000 single-line decodes each, every Record checked)."""
    data, offs = native.generate(native.FMT_RFC5424, 4242, 4000, bad_frac=0.02)
    lines = [bytes(data[offs[i]:offs[i + 1]]) for i in range(4000)]
    obuf, ooffs = oracle.decode_dump(0, data, offs)
    want = [obuf[ooffs[i]:ooffs[i + 1]] for i in range(4000)]
    got = native.clone_decode_threads(native.FMT_RFC5424, lines, nthreads=2)
    assert got == want
