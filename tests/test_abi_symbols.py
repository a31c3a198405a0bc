"""The C-ABI library loads on a CPU-only box and exports every symbol include/flowgger_cuda.h declares.
No compute call is made here (there is no GPU and there is no CPU fallback)."""
import ctypes
import json
import re
from pathlib import Path

REPO = Path(__file__).resolve().parent.parent


def declared_functions():
    text = (REPO / "include" / "flowgger_cuda.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"static inline[^{]*\{.*?\n\}", "", text, flags=re.S)  # header-only span helpers (fg_row5424_*) are not exports
    return sorted(set(re.findall(r"\b(fg_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported(native):
    lib = native.load_cuda()
    names = declared_functions()
    assert len(names) >= 14
    for n in names:
        assert hasattr(lib, n), f"{n} declared in flowgger_cuda.h but not exported"


def test_error_strings_match_reference_text(native):
    # every status maps to the exact &'static str of the reference decoders (cited in fg_abi.cu)
    es = {native.error_string(0, s) for s in range(1, native.load_cuda().fg_error_count())} - {None}
    for must in ["Unsupported BOM", "The priority should be inside brackets", "Invalid priority", "Missing version",
                 "Unsupported version", "Missing timestamp",
                 "Unable to parse the date from RFC3339 to Unix time in RFC5424 decoder", "Missing hostname",
                 "Missing application name", "Missing process id", "Missing message id", "Missing message data",
                 "Missing log message", "Malformated RFC5424 message", "Missing structured data",
                 "Format error in the structured data", "Missing ] after structured data",
                 "Unable to parse the English to Unix timestamp in LTSV decoder", "Invalid severity level",
                 "Severity level should be <= 7", "Type error; boolean was expected", "Type error; f64 was expected",
                 "Type error; i64 was expected", "Type error; u64 was expected",
                 "Invalid GELF input, unable to parse as a JSON object", "Empty GELF input", "Invalid GELF timestamp",
                 "GELF host name must be a string", "GELF short message must be a string",
                 "GELF full message must be a string", "GELF version must be a string", "Unsupported GELF version",
                 "Invalid severity level (too high)", "Invalid value type in structured data",
                 "Malformed RFC3164 event: Invalid priority", "Malformed RFC3164 event: Invalid timestamp or hostname",
                 "Invalid time format", "Unable to parse RFC3164 date with year", "Unable to parse the date in RFC3164 decoder"]:
        assert must in es, must
    assert native.error_string(0, 0) is None


def test_reference_strings_present_in_reference_sources():
    """Guard against typos: each error string must be one of the messages of the reference's decoders and line splitter
    (tests/golden/reference_error_strings.json, taken from the reference sources)."""
    import flowgger_b200 as fb
    golden = json.loads((REPO / "tests" / "golden" / "reference_error_strings.json").read_text())
    messages = {m for ms in golden["messages"].values() for m in ms}
    assert "Invalid UTF-8 input" in messages and len(messages) >= 50
    for s in range(1, fb.load_cuda().fg_error_count()):
        e = fb.error_string(0, s)
        if e and not e.startswith("(the reference panics here"):  # FG_E3_PANIC is this repo's name for a reference panic
            assert e in messages, e


def test_no_cpu_fallback_without_gpu(native):
    """On a box without a GPU the decoder must refuse to exist (fail loudly), never parse on the CPU."""
    import torch
    if torch.cuda.is_available():
        return
    import pytest
    with pytest.raises(RuntimeError, match="no CUDA device|fg_create"):
        native.BatchDecoder(native.FMT_RFC5424)


def test_build_info_names_sm100a(native):
    assert "sm_100a" in native.build_info()


def test_generator_is_deterministic(native):
    b1, o1 = native.generate(native.FMT_RFC5424, 5424, 2000)
    b2, o2 = native.generate(native.FMT_RFC5424, 5424, 2000, nthreads=3)
    assert (b1 == b2).all() and (o1 == o2).all()
    b3, o3 = native.generate(native.FMT_RFC5424, 5424, 1000, first_index=1000)
    assert bytes(b1[o1[1000]:]) == bytes(b3)
