"""sjb200_launch_count is documented as the number of kernels the context has launched (include/simdjson_b200.h).  For every
stage-2 entry point, one call's kernels are counted with torch.profiler (kernels only: memsets and copies are not launches)
and compared with the change of the counter.

The entry points are called through ctypes, and every buffer is allocated before the profiled window: a torch fill kernel
inside it would be counted as well."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

DOC = b'{"a": [1, 2.5, "x\\n", true, null, []], "b": {"c": -7, "d": "\\u00e9", "e": {}}}'
NDJSON = b'{"id": 1, "v": [1, 2]}\n{"id": 2, "v": "s"}\n[1, 2, 3]\n{"id": tru}\n7\n{"id": 4, "v": {"w": 0.5}}\n'
POINTERS = ["/id", "/v/0", "", "/v/w"]


@pytest.fixture(scope="module")
def parser():
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    p = DomParserImplementation(0, max_len=1 << 20)
    yield p
    p.close()


def kernels_run(p, call) -> tuple[int, int, list]:
    """(the call's return code, the change of sjb200_launch_count, the names of the kernels the profiler saw)"""
    L, ctx = p._lib, p._ctx
    torch.cuda.synchronize()
    before = L.sjb200_launch_count(ctx)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]) as prof:
        rc = call()
        assert L.sjb200_sync(ctx) == 0
        torch.cuda.synchronize()
    counted = L.sjb200_launch_count(ctx) - before
    names = [e.name for e in prof.events()
             if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith(("Memcpy", "Memset"))]
    return rc, counted, names


class Device:
    """`data` indexed by stage 1 on the parser's context, and every device buffer a stage-2 call on it writes."""

    def __init__(self, p, data: bytes):
        assert p.stage1(data) == 0
        n = self.n = p.n_structural_indexes
        self.p, self.L, self.ctx = p, p._lib, p._ctx
        dev = lambda k, dt: torch.zeros(k, dtype=dt, device="cuda")   # noqa: E731
        self.d_in = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda()
        self.d_idx = torch.from_numpy(p.structural_indexes[: n + 3].view(np.int32).copy()).cuda()
        self.kind, self.err = dev(n, torch.uint8), dev(n, torch.uint8)
        self.val, self.off = dev(n, torch.int64), dev(n, torch.int64)
        self.sb, self.psum = dev(len(data) + 2 * n + 64, torch.uint8), dev(4, torch.int64)
        self.tape, self.sum = dev(4 * n, torch.int64), dev(4, torch.int64)
        self.first, self.dtape, self.dstat = dev(n + 1, torch.int32), dev(n + 1, torch.int64), dev(n, torch.int64)
        k = len(POINTERS)
        self.ctype, self.ccode, self.cval = dev(k * n, torch.uint8), dev(k * n, torch.uint8), dev(k * n, torch.int64)
        torch.cuda.synchronize()

    def primitives(self, strings: bool = True) -> int:
        return self.L.sjb200_stage2_primitives_device_async(
            self.ctx, self.d_in.data_ptr(), self.d_in.numel(), self.d_idx.data_ptr(), self.n, self.kind.data_ptr(), self.err.data_ptr(),
            self.val.data_ptr(), self.off.data_ptr(), self.sb.data_ptr() if strings else None, self.sb.numel(), self.psum.data_ptr())

    def walk(self) -> int:
        return self.L.sjb200_stage2_tape_device_async(
            self.ctx, self.d_in.data_ptr(), self.d_in.numel(), self.d_idx.data_ptr(), self.n, self.kind.data_ptr(), self.err.data_ptr(),
            self.val.data_ptr(), self.off.data_ptr(), self.tape.data_ptr(), self.tape.numel(), self.sum.data_ptr())

    def stream(self) -> int:
        return self.L.sjb200_stage2_stream_device_async(
            self.ctx, self.d_in.data_ptr(), self.d_in.numel(), self.d_idx.data_ptr(), self.n, self.kind.data_ptr(), self.err.data_ptr(),
            self.val.data_ptr(), self.off.data_ptr(), self.tape.data_ptr(), self.tape.numel(), self.first.data_ptr(), self.dtape.data_ptr(),
            self.dstat.data_ptr(), self.sum.data_ptr())


def check(p, call):
    rc, counted, names = kernels_run(p, call)
    assert rc == 0
    assert len(names) > 0
    assert counted == len(names), names


@pytest.mark.parametrize("strings", [True, False])
def test_primitives(parser, strings):
    d = Device(parser, DOC)
    check(parser, lambda: d.primitives(strings))


def test_single_walk(parser):
    d = Device(parser, DOC)
    assert d.primitives() == 0
    check(parser, d.walk)


def test_stream_walk(parser):
    d = Device(parser, NDJSON)
    assert d.primitives() == 0
    check(parser, d.stream)


def test_at_pointers_device(parser):
    from mojo_simdjson_b200.device import pointer_program

    d = Device(parser, NDJSON)
    assert d.primitives() == 0 and d.stream() == 0
    s, ps = d.sum.cpu().tolist(), d.psum.cpu().tolist()
    n_docs, tape_len, strbuf_len = s[0], s[2], ps[1]
    assert n_docs == 6
    raw, offs = pointer_program(POINTERS)
    check(parser, lambda: d.L.sjb200_at_pointers_device_async(
        d.ctx, d.tape.data_ptr(), tape_len, d.sb.data_ptr(), strbuf_len, d.dtape.data_ptr(), d.dstat.data_ptr(), n_docs, raw, offs, len(POINTERS),
        d.ctype.data_ptr(), d.ccode.data_ptr(), d.cval.data_ptr()))


def host_outputs(n: int, length: int):
    return (np.zeros(4 * n, np.uint64), np.zeros(length + 2 * n + 64, np.uint8), np.zeros(n + 1, np.uint32), np.zeros(n + 1, np.uint64),
            np.zeros(n, np.uint64))


def test_stage2_host(parser):
    assert parser.stage1(DOC) == 0
    tape, sb, _, _, _ = host_outputs(parser.n_structural_indexes, len(DOC))
    tl, sl, inexact = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    check(parser, lambda: parser._lib.sjb200_stage2(parser._ctx, tape.ctypes.data, tape.size, sb.ctypes.data, sb.size, C.byref(tl), C.byref(sl),
                                                    C.byref(inexact)))


def test_stage2_stream_host(parser):
    assert parser.stage1(NDJSON) == 0
    n = parser.n_structural_indexes
    tape, sb, first, doc_tape, status = host_outputs(n, len(NDJSON))
    nd, nf, tl, sl, inexact = (C.c_uint64(0) for _ in range(5))
    check(parser, lambda: parser._lib.sjb200_stage2_stream(parser._ctx, tape.ctypes.data, tape.size, sb.ctypes.data, sb.size, first.ctypes.data,
                                                           doc_tape.ctypes.data, status.ctypes.data, n, C.byref(nd), C.byref(nf), C.byref(tl),
                                                           C.byref(sl), C.byref(inexact)))
    assert nd.value == 6 and nf.value == 1


def test_stage2_stream_at_pointers_host(parser):
    from mojo_simdjson_b200.device import pointer_program

    assert parser.stage1(NDJSON) == 0
    n = parser.n_structural_indexes
    _, sb, _, _, _ = host_outputs(n, len(NDJSON))
    cells = len(POINTERS) * n
    ty, code, val = np.zeros(cells, np.uint8), np.zeros(cells, np.uint8), np.zeros(cells, np.int64)
    raw, offs = pointer_program(POINTERS)
    nd, sl = C.c_uint64(0), C.c_uint64(0)
    check(parser, lambda: parser._lib.sjb200_stage2_stream_at_pointers(parser._ctx, raw, offs, len(POINTERS), ty.ctypes.data, code.ctypes.data,
                                                                       val.ctypes.data, cells, sb.ctypes.data, sb.size, C.byref(nd), C.byref(sl)))
    assert nd.value == 6
