"""Pin the C restatement (oracle/c/b9_oracle.c) to the Python oracle, whose Python halves are the
reference's own stdlib calls. Every task: same status, same result bytes, same queue wire bytes."""
import base64
import json
import random

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

from beta9_b200 import synth
from oracle import coracle
from oracle.pyoracle import loop

PY2C = {"COMPLETE": coracle.COMPLETE, "ERROR": coracle.ERROR, "REJECTED": coracle.REJECTED}


def compare(batch, handler, allow_unsupported=False):
    r = coracle.run_batch(batch.task_ids, batch.payload, batch.offsets, handler, keep_wire=True)
    pr = loop.run_task_loop(batch.tasks(), [bytes(x) for x in batch.task_ids], handler, keep_wire=True)
    n_unsup = 0
    for i, p in enumerate(pr):
        if r.status[i] == coracle.UNSUPPORTED:
            assert allow_unsupported, (i, batch.task(i))
            n_unsup += 1
            continue
        assert PY2C[p.status] == r.status[i], (i, batch.task(i), p.status, r.status[i])
        assert p.result == r.result(i), (i, batch.task(i))
        assert (p.wire or b"") == r.wire_msg(i), (i, batch.task(i))
    return n_unsup


def test_identity_strings_with_adversarial():
    compare(synth.strings_batch(3000, 64, adversarial_frac=0.3), "identity")
    compare(synth.strings_batch(500, 256, adversarial_frac=0.5, seed=7), "crc32")


def test_crc_zipf():
    compare(synth.crc_batch(3000), "crc32")
    compare(synth.crc_batch(500, seed=3), "identity")


def test_vadd():
    compare(synth.vadd_batch(2000), "vadd_f32")
    compare(synth.vadd_batch(300, floats_per_vec=5, seed=1), "vadd_f32")
    # (NaN payloads, infinities, denormals: test_vadd_two_nan_operands)


def test_vadd_two_nan_operands():
    """What the reference's arithmetic (numpy `a + b` on this x86-64 host) leaves open: when BOTH operands of an
    element are NaN, the quieted payload that survives is the first operand's inside numpy's SIMD body and the second's
    in its scalar tail, i.e. it depends on the element's position and the vector length. Everything else — one NaN
    operand, inf + -inf, denormals, overflow — is position-independent. The C oracle (and the device) always return the
    first operand, quieted; this test pins exactly that much: equal to numpy everywhere except two-NaN elements, where
    numpy's answer must be one of the two quieted operands."""
    import base64
    import json as _json
    from oracle.pyoracle import handlers
    two_nan = differing = 0
    for fpv in list(range(1, 41)) + [64, 100]:
        b = synth.vadd_special_batch(8, floats_per_vec=fpv, seed=1000 + fpv)
        o = coracle.run_batch(b.task_ids, b.payload, b.offsets, "vadd_f32")
        for i in range(b.n):
            s = _json.loads(b.task(i))["args"][0]
            raw = np.frombuffer(base64.b64decode(s), "<u4")
            n = raw.size // 2
            x, y = raw[:n], raw[n:]
            ref = np.frombuffer(base64.b64decode(handlers.vadd_f32(s)), "<u4")           # numpy
            got = np.frombuffer(base64.b64decode(o.result(i)[1:-1]), "<u4")              # C oracle
            xn, yn = (x & 0x7FFFFFFF) > 0x7F800000, (y & 0x7FFFFFFF) > 0x7F800000
            both = xn & yn
            assert np.array_equal(got[~both], ref[~both]), (fpv, i)
            assert np.array_equal(got[both], x[both] | 0x00400000)
            assert np.all((ref[both] == (x[both] | 0x00400000)) | (ref[both] == (y[both] | 0x00400000)))
            two_nan += int(both.sum())
            differing += int((got[both] != ref[both]).sum())
    assert two_nan > 100            # (differing may be 0 on a host whose numpy has no scalar tail; here it is not)


def test_json_sum():
    compare(synth.json_batch(500), "json_sum")
    compare(synth.json_batch(100, doc_bytes=300, seed=2), "identity")


def test_json_sum_near_the_int64_limits():
    """Sums of |s| in (2^62, 2^64) in both signs, of random values below 2^53 (exact in float64): the C oracle prints
    every sum inside int64 exactly as Python does, and declines only the ones outside."""
    rng = random.Random(62)
    totals = [2**62 + 1, 2**63 - 2, 2**63 - 1, 2**63, 2**63 + 1, 2**64 - 1] + [rng.randrange(2**62, 2**63) for _ in range(20)]
    payloads, outside = [], 0
    for t in totals + [-t for t in totals]:
        vals, left = [], t
        while abs(left) > 2**53:
            v = rng.randrange(2**52, 2**53) * (1 if left > 0 else -1)
            vals.append(v)
            left -= v
        vals.append(left)
        rng.shuffle(vals)
        payloads.append(loop.sdk_put_payload({"values": vals}))
        outside += not -2**63 <= t < 2**63
    assert compare(synth.from_payloads(payloads), "json_sum", allow_unsupported=True) == outside


HANDCRAFTED = [
    b'{"args": ["x"], "kwargs": {}}', b'{"args":["x"]}', b' { "kwargs" : { } , "args" : [ "x" ] } ',
    b'{"args": [""], "kwargs": {}}', b'{"args": [], "kwargs": {}}', b'{"args": ["a", "b"], "kwargs": {}}',
    b'{"args": ["a"], "kwargs": {"k": 1}}', b'{"args": ["a"], "kwargs": null}', b'{"args": null}', b"null", b"{}",
    b"[]", b'"x"', b"", b"{", b'{"args": ["x"],}', b'{"args": ["\\ud83d"]}', b'{"args": ["\\ud83d\\ude00"]}',
    b'{"args": ["\\ude00\\ud83d"]}', b'{"args": ["\xff"]}', b'{"args": ["\xc3\xa9\xe2\x80\xa8"]}',
    b'{"args": ["\\u0000\\u001f\\u007f\\u0080\\u2028\\uffff"]}', b'{"args": ["<>&/\\/"]}',
    b'{"args": ["\x01"]}', b'{"args": ["\\q"]}', b'{"ARGS": ["up"]}', b'{"args": ["1"], "args": ["2"]}',
    b'{"kwargs": {"a": 1}, "kwargs": {}, "args": ["x"]}', b'{"args": [0]}', b'{"args": [-0]}', b'{"args": [1.0]}',
    b'{"args": [1e3]}', b'{"args": [1.5]}', b'{"args": [9007199254740992]}', b'{"args": [9007199254740994]}',
    b'{"args": [1e999]}', b'{"x": 1e999, "args": ["ok"]}', b'{"args": [true]}', b'{"args": [false]}',
    b'{"args": [null]}', b'{"args": [[]]}', b'{"args": [{}]}', b'{"args": [[1, "a", null, true, {"b": [], "a": "<"}]]}',
    b'{"args": [{"b": 1, "a": 2, "b": 3}]}', b'{"args": [{"values": [1, 2, 3]}]}', b'{"args": [{"values": []}]}',
    b'{"args": [{"values": [true, 2]}]}', b'{"args": [{"values": [1, "a"]}]}', b'{"args": [{"values": "ab"}]}',
    b'{"args": [{"values": ""}]}', b'{"args": [{"values": {}}]}', b'{"args": [{"values": {"a": 1}}]}',
    b'{"args": [{"values": null}]}', b'{"args": [{"valuez": [1]}]}', b'{"args": [{"values": [1], "values": [5, 6]}]}',
    b'{"args": [{"valu\\u0065s": [4]}]}', b'{"args": [{"values": [-5, 5]}]}', b'{"args": [{"values": [1.5]}]}',
    b'{"args": [{"values": [[1]]}]}', b'{"args": [[1, 2]]}', b'{"args": ["AAAA"]}', b'{"args": ["AAA="]}',
    b'{"args": ["AA=="]}', b'{"args": ["A==="]}', b'{"args": ["AAA"]}', b'{"args": ["AA\\nAA"]}', b'{"args": ["=AAA"]}',
    b'{"args": ["AAAAAAAAAAA="]}', b'{"args": ["AAAAAAAAAAAAAAAAAAAAAA=="]}', b'{"args": ["AB==AAAA"]}',
    b'{"args": ["A-AA"]}', b'{"args": ["\\u00e9AAA"]}', b'{"args": ["QUJDREVGR0g="]}', b'{"args": ["AAAAAAAAAAB="]}',
    # a number that overflows float64 inside a DECODED value refuses the payload even if a later duplicate of the key
    # overwrites it (decode.go keeps the first conversion error); under an unknown key it is never converted
    b'{"args": [1e999], "args": ["x"]}', b'{"args": [{"k": 5e08858}], "\\u0061rgs": []}', b'{"kwargs": {"a": 1e999, "a": 1}, "args": ["x"]}',
    b'{"args": ["x"], "kwargs": {"a": 1e999}, "kwargs": {"a": 2}}', b'{"args": ["x"], "other": 1e999, "other": 1}', b'{"args": 1e999, "args": ["x"]}',
    # json_sum at -2^63, 2^63 - 1 (the int64 limits: decided, printed exactly) and 2^63 (beyond: the C oracle declines)
    # as sums of 2^53 = 9007199254740992, the largest power of two whose neighbours float64 still holds exactly
    b'{"args": [{"values": [' + b", ".join([b"-9007199254740992"] * 1024) + b']}], "kwargs": {}}',
    b'{"args": [{"values": [' + b", ".join([b"9007199254740992"] * 1023 + [b"9007199254740991"]) + b']}], "kwargs": {}}',
    b'{"args": [{"values": [' + b", ".join([b"9007199254740992"] * 1024) + b']}], "kwargs": {}}',
]


@pytest.mark.parametrize("handler", ["identity", "crc32", "vadd_f32", "json_sum"])
def test_handcrafted(handler):
    compare(synth.from_payloads(HANDCRAFTED), handler, allow_unsupported=True)


def test_handcrafted_unsupported_is_only_floats():
    b = synth.from_payloads(HANDCRAFTED)
    r = coracle.run_batch(b.task_ids, b.payload, b.offsets, "identity")
    unsup = {HANDCRAFTED[i] for i in range(b.n) if r.status[i] == coracle.UNSUPPORTED}
    assert unsup == {b'{"args": [1.5]}', b'{"args": [9007199254740994]}', b'{"args": [{"values": [1.5]}]}'}


# ---- fuzz: arbitrary JSON documents as args / kwargs, serialised the way the SDK does
json_leaf = st.one_of(st.none(), st.booleans(), st.integers(-2**53, 2**53),
                      st.text(max_size=12), st.text(alphabet='"\\<>&/\n\t\x00\x7fé 😀\U0001f600ab', max_size=8))
json_val = st.recursive(json_leaf, lambda c: st.one_of(st.lists(c, max_size=4),
                                                      st.dictionaries(st.text(max_size=5), c, max_size=4)), max_leaves=12)


@settings(max_examples=300, deadline=None, suppress_health_check=list(HealthCheck))
@given(st.lists(st.tuples(st.lists(json_val, max_size=2), st.dictionaries(st.text(max_size=4), json_val, max_size=1)),
                min_size=1, max_size=6), st.sampled_from(["identity", "crc32", "vadd_f32", "json_sum"]))
def test_fuzz_sdk_payloads(tasks, handler):
    payloads = [loop.sdk_put_payload(*a, **{k: v for k, v in kw.items()}) for a, kw in tasks]
    compare(synth.from_payloads(payloads), handler)


@settings(max_examples=300, deadline=None, suppress_health_check=list(HealthCheck))
@given(st.lists(st.binary(max_size=40), min_size=1, max_size=6), st.sampled_from(["identity", "crc32"]))
def test_fuzz_raw_bytes_in_string(blobs, handler):
    # arbitrary bytes (invalid UTF-8, stray quotes, control bytes) between the canonical frame
    payloads = [synth.PREFIX + b + synth.SUFFIX for b in blobs]
    compare(synth.from_payloads(payloads), handler, allow_unsupported=True)


def test_fuzz_mutations():
    rnd = random.Random(0xB9)
    base = [loop.sdk_put_payload("hello \"w\" \\ é"), loop.sdk_put_payload({"values": [1, 2, 3], "id": 7}),
            loop.sdk_put_payload(base64.b64encode(bytes(range(64))).decode())]
    payloads = []
    for _ in range(3000):
        p = bytearray(rnd.choice(base))
        for _ in range(rnd.randint(1, 3)):
            k = rnd.randrange(len(p))
            op = rnd.random()
            if op < 0.4:
                p[k] = rnd.randrange(256)
            elif op < 0.7:
                del p[k]
            else:
                p.insert(k, rnd.choice(b'"\\{}[],: \x00\xffu0'))
        payloads.append(bytes(p))
    b = synth.from_payloads(payloads)
    for h in ("identity", "crc32", "vadd_f32", "json_sum"):
        compare(b, h, allow_unsupported=True)


def test_threads_give_same_answer():
    b = synth.strings_batch(5000, 64, adversarial_frac=0.2)
    r1 = coracle.run_batch(b.task_ids, b.payload, b.offsets, "identity", nthreads=1)
    r4 = coracle.run_batch(b.task_ids, b.payload, b.offsets, "identity", nthreads=4)
    assert np.array_equal(r1.status, r4.status) and np.array_equal(r1.offsets, r4.offsets)
    assert np.array_equal(r1.payload, r4.payload)
