"""CPU-only checks of the drop-in boundary: the library builds, loads and exports what the header declares."""
import os
import re

from mojo_simdjson_b200 import _native, build, errors

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "simdjson_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sjb200_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_exports_every_declared_symbol():
    build.build_cuda()
    L = _native.lib()
    names = _declared()
    assert len(names) >= 20
    for name in names:
        assert hasattr(L, name), f"{name} declared in include/simdjson_b200.h but not exported"
        assert name in _native.SIGNATURES, f"{name} has no ctypes signature"
    assert L.sjb200_version() == 1


def test_error_codes_match_reference_values():
    # reference src/mojo_simdjson/errors.mojo:2-34
    assert (errors.SUCCESS, errors.CAPACITY, errors.MEMALLOC, errors.UTF8_ERROR) == (0, 1, 2, 11)
    assert (errors.EMPTY, errors.UNESCAPED_CHARS, errors.UNCLOSED_STRING, errors.UNEXPECTED_ERROR) == (13, 14, 15, 24)
    assert errors.NUM_ERROR_CODES == 32
    hdr = open(os.path.join(ROOT, "include", "simdjson_b200.h")).read()
    for name, val in re.findall(r"#define SJB200_([A-Z0-9_]+) (\d+)\s", hdr):
        if hasattr(errors, name):
            assert getattr(errors, name) == int(val)


def test_host_splitter_without_gpu():
    import ctypes as C

    L = _native.lib()
    data = b'{"a":1}\n' * 1000
    offs = (C.c_uint64 * 64)()
    n = C.c_uint32(0)
    rc = L.sjb200_batch_split_host(data, len(data), 1000, offs, 63, C.byref(n))
    assert rc == 0
    cuts = [int(offs[i]) for i in range(n.value + 1)]
    assert cuts[0] == 0 and cuts[-1] == len(data)
    for a, b in zip(cuts, cuts[1:]):
        assert 0 < b - a <= 2000 and data[b - 1:b] == b"\n"
    # a window without a newline cannot be cut
    rc = L.sjb200_batch_split_host(b"x" * 5000, 5000, 1000, offs, 63, C.byref(n))
    assert rc == errors.CAPACITY


def test_no_gpu_means_loud_failure_not_fallback():
    import pytest

    L = _native.lib()
    if L.sjb200_device_count() > 0:
        pytest.skip("a GPU is present")
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    with pytest.raises(RuntimeError):
        DomParserImplementation(0)
