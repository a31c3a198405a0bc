"""Result-table overflow, regrow and redo through every batch entry point of the C ABI, for every format, against the
oracle.  The contexts are small (max_batch_bytes = 256 KiB, so every side table starts small) and take 128 lines per
chunk, so one call spans many chunks; each shaped batch overflows one table.  GPU only."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

R5, LT, GE, R3 = 0, 1, 2, 3
YEAR = 2026
MAX_BYTES = 1 << 18
TS = b"2015-08-05T15:53:45.637824Z"


def _sd_pairs(k):
    return b"<13>1 " + TS + b" h a p m [i" + b"".join(b' k%02d="vvvv"' % j for j in range(k)) + b"] m"


def _quotes(k):
    return b"<13>1 " + TS + b" h a p m - " + b'\\"' * k


# first sizes at 256 KiB: RFC5424 e8 11008 rows, arena 64 KiB, wide 1024 rows, wide entries 4096 rows;
# LTSV / GELF entries 11008 rows; RFC3164 arena 64 KiB
SHAPED = {
    R5: {
        "e8": [_sd_pairs(50)] * 240,                                                              # ~13000 8-byte rows
        "arena": [b"<13>1 " + TS + b' h a p m [e v="' + b"x" * 190 + b'\\"y"] m'] * 360,        # ~70 KiB unescaped
        "wide": [b"<13>1 " + TS + b' h a p m [id  a="1" b="2" c="3"] m'] * 1100,                # slow path: 1100 rows, 4400 entries
    },
    LT: {"entries": [b"time:[5/Aug/2015:15:53:45 +0000]\thost:h\t" +
                     b"\t".join(b"%c%c:1" % (97 + j // 26, 97 + j % 26) for j in range(60))] * 200},
    GE: {"entries": [b'{"version":"1.1","host":"h","short_message":"m",' +
                     b",".join(b'"_%c%c":1' % (97 + j // 26, 97 + j % 26) for j in range(60)) + b"}"] * 200},
    R3: {"arena": [b"<13>Aug  6 11:15:24 host tag: " + b"x y  " * 40] * 440},                  # re-joined messages
}


def _batch(native, oracle, fmt, shaped, seed):
    n_gen = 100 if fmt == GE else 300
    d, o = native.generate(fmt, seed, n_gen)
    lines = [bytes(d[o[i]:o[i + 1]]).replace(b"\n", b" ").replace(b"\r", b" ") for i in range(n_gen)] + shaped
    lines = [l for l in lines if _utf8(l)]  # split mode reports invalid UTF-8 itself: keep the streams comparable
    data, offs = oracle.pack(lines)
    assert len(data) <= MAX_BYTES
    return lines, data, offs


def _utf8(b):
    try:
        b.decode("utf-8")
        return True
    except UnicodeDecodeError:
        return False


def _decoder(native, fmt, **kw):
    kw.setdefault("max_batch_bytes", MAX_BYTES)
    kw.setdefault("max_batch_lines", 1 << 12)
    return native.BatchDecoder(fmt, chunk_lines=128, rfc3164_year=YEAR if fmt == R3 else 0, **kw)


def _oracle_dump(oracle, fmt, data, offs):
    return oracle.decode_dump(fmt, data, offs, oracle.Rfc3164Config(YEAR) if fmt == R3 else None, nthreads=8)


def _run(dec, how, lines, data, offs):
    """One call of the entry point -> canonical dumps and dump offsets."""
    if how == "decode":
        return dec.dump(dec.decode(data, offs), data, offs)
    if how == "split":
        stream = np.frombuffer(b"".join(l + b"\n" for l in lines), dtype=np.uint8).copy()
        buf, bo, line_offs, _ = dec.split_dump(stream)
        assert len(line_offs) == len(lines) + 1
        return buf, bo
    dec.upload(data, offs)
    dec.parse_resident()
    return dec.dump(dec.download(), data, offs)


def _launches(dec, how, lines, data, offs):
    n0 = dec.kernel_launches()
    got = _run(dec, how, lines, data, offs)
    return got, dec.kernel_launches() - n0


@pytest.mark.parametrize("how", ["decode", "split", "resident"])
@pytest.mark.parametrize("fmt", [R5, LT, GE, R3])
def test_table_regrow_and_redo(native, oracle, fmt, how):
    dec = _decoder(native, fmt)
    try:
        for seed, (table, shaped) in enumerate(SHAPED[fmt].items()):
            lines, data, offs = _batch(native, oracle, fmt, shaped, seed)
            want = _oracle_dump(oracle, fmt, data, offs)
            first, d1 = _launches(dec, how, lines, data, offs)
            again, d2 = _launches(dec, how, lines, data, offs)
            assert d1 == 2 * d2, f"{table}: the first call should have regrown the table and redone the batch"
            for buf, bo in (first, again):
                assert buf == want[0] and np.array_equal(bo, want[1]), f"{table}: differs from the oracle"
    finally:
        dec.close()


def test_encoder_regrows_side_table_and_output(native, oracle):
    """One fused decode + encode call whose 8-byte SD rows overflow their table and whose records overflow the output
    buffer (2 x max_batch_bytes + 200 bytes per line at first): both regrow, and the records equal the oracle's."""
    d, o = native.generate(R5, 7, 30)
    lines = [bytes(d[o[i]:o[i + 1]]) for i in range(30)]
    lines += [_sd_pairs(50)] * 120 + [_quotes(280)] * 80   # ~6200 rows over 5632; JSON ~4x the quoted input
    data, offs = oracle.pack(lines)
    dec = _decoder(native, R5, max_batch_bytes=1 << 17, max_batch_lines=256)
    try:
        assert len(data) <= 1 << 17
        n0 = dec.kernel_launches()
        buf, eo, _, _ = dec.decode_encode_gelf(data, offs)
        d1 = dec.kernel_launches() - n0
        wbuf, wo = oracle.decode_encode_gelf(R5, data, offs)
        assert buf == wbuf and np.array_equal(eo, wo)
        assert int(eo[-1]) > 2 * (1 << 17) + 256 * 200
        n0 = dec.kernel_launches()
        buf, eo, _, _ = dec.decode_encode_gelf(data, offs)
        assert d1 == 2 * (dec.kernel_launches() - n0)  # one redo regrew both
        assert buf == wbuf and np.array_equal(eo, wo)
        assert int(dec.decode(data, offs).raw.n_entries8) > 5632  # the first size of the 8-byte row table
    finally:
        dec.close()
