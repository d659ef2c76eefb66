"""The DEVICE JSON parser (beta9_b200/csrc/json_device.cuh), compiled for the host by
tests/host_shim/host_parse.cpp, against the oracle on a CPU: what it accepts / refuses, how many
arguments it finds, whether keyword arguments are present, and which token it takes for args[0] —
under the SDK-payload rules (struct decode) and under B9_TF_HTTP_BODY (SerializeHttpPayload's map
rules). The kernels' own tests need a GPU; this one runs everywhere and sees the same source."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from oracle.pyoracle.gojson import GoJSONError, go_unmarshal, go_unmarshal_task_payload
from oracle.pyoracle.httpserialize import InvalidRequestPayload, serialize_http_payload

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host_shim", "host_parse.cpp")
SO = os.path.join(HERE, "host_shim", "libhostparse.so")
GXX = os.environ.get("CXX", "g++")


@pytest.fixture(scope="module")
def parser():
    return load_host_shim()


def load_host_shim():
    """Builds (when a source is newer) and loads the host shim; returns parse(b, http) with .run, .transcode, .rfc3339
    and .vadd_fast attached. Skips the calling test where there is no host C++ compiler."""
    csrc = os.path.join(os.path.dirname(HERE), "beta9_b200", "csrc")
    deps = [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".h"))]
    if not os.path.exists(SO) or os.path.getmtime(SO) < max([os.path.getmtime(SRC)] + [os.path.getmtime(d) for d in deps]):
        r = subprocess.run([GXX, "-O2", "-std=c++17", "-shared", "-fPIC", "-o", SO, SRC], capture_output=True, text=True)
        if r.returncode:
            pytest.skip("no host C++ compiler for the shim: " + r.stderr[-300:])
    lib = C.CDLL(SO)
    lib.b9_host_parse.argtypes = [C.c_char_p, C.c_uint32, C.c_int, C.POINTER(C.c_uint32)]
    lib.b9_host_run.argtypes = [C.c_char_p, C.c_uint32, C.c_int, C.c_int, C.POINTER(C.c_uint8), C.POINTER(C.c_uint8), C.c_char_p, C.c_uint32]
    lib.b9_host_run.restype = C.c_long

    def parse(b: bytes, http: bool):
        out = (C.c_uint32 * 12)()
        lib.b9_host_parse(b, len(b), 1 if http else 0, out)
        return list(out)

    def run(b: bytes, http: bool, handler: int):
        st, has = C.c_uint8(0), C.c_uint8(0)
        buf = C.create_string_buffer(8 * len(b) + 64)
        n = lib.b9_host_run(b, len(b), 1 if http else 0, handler, C.byref(st), C.byref(has), buf, len(buf))
        assert n >= 0
        return int(st.value), (buf.raw[:n] if has.value else None)
    lib.b9_host_go_transcode.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32]
    lib.b9_host_go_transcode.restype = C.c_long
    lib.b9_host_rfc3339nano.argtypes = [C.c_longlong, C.c_char_p]
    lib.b9_host_rfc3339nano.restype = C.c_long

    def transcode(tok: bytes):
        buf = C.create_string_buffer(8 * len(tok) + 64)
        n = lib.b9_host_go_transcode(tok, len(tok), buf, len(buf))
        return None if n < 0 else buf.raw[:n]

    def rfc3339(ns: int) -> bytes:
        buf = C.create_string_buffer(64)
        n = lib.b9_host_rfc3339nano(ns, buf)               # (call first: `buf.raw` is a snapshot)
        return buf.raw[:n]
    lib.b9_host_vadd_fast.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32]
    lib.b9_host_vadd_fast.restype = C.c_long

    def vadd_fast(b: bytes):
        buf = C.create_string_buffer(len(b) + 64)
        n = lib.b9_host_vadd_fast(b, len(b), buf, len(buf))
        assert n >= -1, n                                # -2..-5: the fast path contradicted itself
        return None if n < 0 else buf.raw[:n]
    parse.vadd_fast = vadd_fast
    parse.run, parse.transcode, parse.rfc3339 = run, transcode, rfc3339
    return parse


def _oracle(b: bytes, http: bool):
    try:
        args, kwargs = serialize_http_payload(b) if http else go_unmarshal_task_payload(b)
    except (GoJSONError, InvalidRequestPayload):
        return None
    return list(args or []), dict(kwargs or {})


def _payloads():
    from beta9_b200 import synth
    from tests.test_oracle_c_vs_py import HANDCRAFTED
    from tests.test_oracle_reference_answers import SERIALIZE_CASES
    out = list(HANDCRAFTED) + [c[1].encode() for c in SERIALIZE_CASES]
    out += [b'{"args": ["abc"]}', b'{"x": 1}', b'', b'  \n', b'null', b' null ', b'[1]', b'"s"', b'7', b'{"args": "notalist"}', b'{"args": null}',
            b'{"args": ["a"], "kwargs": 5}', b'{"args": ["a"], "kwargs": null}', b'{"args": ["a"], "other": [1e999]}', b'{"\\u0061rgs": ["esc"]}',
            b'{"Args": ["folded?"]}', b'{"ARGS": ["x"], "KWARGS": {}}', b'{"args": ["a"], "args": 1}', b'{"args": 1, "args": ["last"]}',
            b'{"kwargs": {"k": 1}, "kwargs": {}, "args": ["dup kw"]}', b'{"kwargs": {}, "kwargs": {"k": 1}, "args": ["dup kw 2"]}',
            b'{"args": ["x"], "kwargs": {}, "extra": true}', b'{"args": ["x"], "extra": true}', b'{"k\\u0077args": {}, "args": ["esc key"]}',
            b'{"kwargs": 1, "kwargs": {}, "args": [1]}', b'{"kwargs": {}, "kwargs": 1, "args": [1]}', b'{"a": 1e400}', b'{"args": [1], "a": {"b": 1e400}}',
            b'{"\\u212aargs": [1]}', b'{"arg\\u017f": [1]}', b'{"args": [1, 2.5, true, null, "s", {"a": []}, [1]]}']
    for b in (synth.strings_batch(40, 48, adversarial_frac=0.4, seed=3), synth.json_batch(4, doc_bytes=200), synth.vadd_batch(4, floats_per_vec=3)):
        out += [b.task(i) for i in range(b.n)]
    rng = np.random.default_rng(20260921)
    alphabet = list(b'{}[],:" 01e.-nulltrackwgsAK\\')
    base = [p for p in out if len(p) >= 4]
    for p in base:
        for _ in range(4):
            m = bytearray(p)
            pos = int(rng.integers(0, len(m)))
            op = int(rng.integers(0, 3))
            ch = int(rng.choice(alphabet))
            if op == 0: m[pos] = ch
            elif op == 1: del m[pos]
            else: m[pos:pos] = bytes([ch])
            out.append(bytes(m))
    return out


@pytest.mark.parametrize("http", [False, True], ids=["sdk_payload", "http_body"])
def test_device_parser_agrees_with_the_oracle(parser, http):
    payloads = _payloads()
    checked = declined = 0
    for b in payloads:
        status, nargs, kw_nonempty, a0_kind, a0_off, a0_len, a0_flags, kw_merged = parser(b, http)[:8]
        want = _oracle(b, http)
        if status == 4:                                   # nesting deeper than the device stack: declined, never decided
            declined += 1
            continue
        if want is None:
            assert status == 3, (b, status)
            continue
        assert status == 0, (b, status, want)
        args, kwargs = want
        assert nargs == len(args), (b, nargs, args)
        if not (kw_merged and not http):                  # (struct rules: merged duplicate kwargs maps are flagged, not resolved)
            assert bool(kw_nonempty) == bool(kwargs), (b, kw_nonempty, kwargs)
        if args:
            tok = b[a0_off:a0_off + a0_len]
            try:
                got0 = go_unmarshal(tok)                  # the token the device would hand to the handler, decoded by Go's rules
            except GoJSONError:                           # (a number Go refuses is refused for the whole payload: covered above)
                raise AssertionError((b, tok))
            assert got0 == args[0] or (got0 != got0 and args[0] != args[0]), (b, tok, got0, args[0])
        checked += 1
    assert checked > len(payloads) // 4 and declined < len(payloads) // 20


@pytest.mark.parametrize("http", [False, True], ids=["sdk_payload", "http_body"])
@pytest.mark.parametrize("handler", ["identity", "crc32", "vadd_f32", "json_sum"])
def test_device_sequential_path_agrees_with_the_oracle(parser, handler, http):
    """parse -> handler -> result bytes of the device's one-thread-per-task path (what every payload outside a
    fast path's domain goes through), against the oracle's task loop."""
    from oracle.pyoracle import loop
    payloads = _payloads()
    ids = [bytes([i & 255]) * 16 for i in range(len(payloads))]
    want = loop.run_task_loop(payloads, ids, handler, http_body=http)
    code = {"COMPLETE": 0, "ERROR": 1, "RETRY": 2, "REJECTED": 3}
    hid = ["identity", "crc32", "vadd_f32", "json_sum"].index(handler)
    declined = 0
    for b, w in zip(payloads, want):
        st, res = parser.run(b, http, hid)
        if st == 4:                                       # outside the device handler's domain: declined, never guessed
            assert res is None
            declined += 1
            continue
        assert st == code[w.status], (b, st, w.status)
        assert res == w.result, (b, res, w.result)
    assert declined < len(payloads) // 5


def test_device_go_value_encoder_agrees_with_the_oracle(parser):
    """go_transcode (wire_encode.cuh): the args list / kwargs object of a TaskMessage re-encoded by Go's rules, and
    the RFC3339Nano `expires`. Wherever the device encoder does not decline, its bytes are the oracle's."""
    from oracle.pyoracle.gojson import go_marshal, go_time_rfc3339nano
    done = declined = 0
    for b in _payloads():
        try:
            args, kwargs = go_unmarshal_task_payload(b)
        except GoJSONError:
            continue
        # the value tokens as they sit in the payload (the spans the device parser reports)
        st = parser(b, False)
        if st[0] != 0 or st[7]:
            continue
        for val, off, ln in ((args, st[8], st[9]), (kwargs, st[10], st[11])):
            if val is None or ln == 0:
                continue
            tok = b[off:off + ln]
            got = parser.transcode(tok)
            if got is None:
                declined += 1
                continue
            assert got == go_marshal(val).encode(), (tok, got, go_marshal(val))
            done += 1
    assert done > 100
    for ns in (0, 1, 999_999_999, 1_000_000_000, 1_789_970_992_573_161_412, 1_709_210_096_000_000_000, 4_102_444_800_000_000_000,
               951_782_400_123_000_000, 1_718_000_000_120_000_000):
        assert parser.rfc3339(ns) == go_time_rfc3339nano(ns).encode(), ns


def test_vadd_fast_path_agrees_with_the_oracle(parser):
    """vadd_f32's branch-free, in-place fast path (vadd_fast.cuh) on the host: every float count 1..70 (all base64
    phases of a, of b and of the padding), raw bit patterns (NaN payloads, inf - inf, denormals), every task
    alignment; whatever it decides must be the oracle's bytes, and canonical payloads must be decided."""
    from beta9_b200 import synth
    payloads, canonical = [], 0
    for fpv in list(range(1, 71)) + [100, 333]:
        for b in (synth.vadd_batch(6, floats_per_vec=fpv, seed=fpv), synth.vadd_special_batch(6, floats_per_vec=fpv, seed=fpv)):
            payloads += [b.task(i) for i in range(b.n)]
    canonical = len(payloads)
    rng = np.random.default_rng(5)
    for p in list(payloads[::7]):                         # corrupted text: must be left to the sequential path or still be right
        m = bytearray(p)
        pos = int(rng.integers(11, len(m) - 17))
        m[pos] = int(rng.choice(list(b"=!-_ \"\\\x7f\xc3")))
        payloads.append(bytes(m))
        m = bytearray(p); del m[pos]; payloads.append(bytes(m))
    # expected bytes: the C oracle (it spells out "a NaN operand comes back quieted, the first one winning"; numpy, the
    # reference's arithmetic, agrees except when BOTH operands are NaN, where its answer depends on the element's position
    # in its SIMD loop: tests/test_oracle_c_vs_py.py::test_vadd_two_nan_operands)
    from oracle import coracle
    b = synth.from_payloads(payloads)
    o = coracle.run_batch(b.task_ids, b.payload, b.offsets, "vadd_f32")
    decided = 0
    for i, p in enumerate(payloads):
        got = parser.vadd_fast(p)
        if got is None:
            assert i >= canonical, p                      # a canonical payload must take the fast path
            continue
        decided += 1
        assert int(o.status[i]) == 0 and got == o.result(i), (p, got, o.result(i))
    assert decided >= canonical
