"""GPU parity: the CUDA drain path through the C ABI against the oracle, bit for bit."""
import numpy as np
import pytest

from beta9_b200 import synth
from oracle import coracle
from tests import golden_util as G

pytestmark = pytest.mark.gpu

HANDLERS = ["identity", "crc32", "vadd_f32", "json_sum"]


@pytest.fixture(scope="module")
def dq():
    from beta9_b200.device_queue import DeviceQueue
    q = DeviceQueue(ring_bytes=1 << 31, ring_tasks=1 << 21, max_drain_tasks=1 << 21, max_result_bytes=3 << 30)
    yield q
    q.close()


def run_gpu(dq, batch, handler):
    assert dq.depth() == 0
    dq.push_batch(batch.task_ids, batch.payload, batch.offsets)
    assert dq.depth() == batch.n
    r = dq.drain(handler, max_tasks=batch.n)
    assert dq.depth() == 0 and r.n_popped == batch.n
    return r


def assert_matches_python_oracle_where_c_declines(batch, r, o, http=False):
    """Tasks the C oracle declines (json_sum outside int64, number literals it does not print) but the device decided:
    the Python oracle's task loop, which is exact everywhere, must give the same status and bytes. Returns how many
    tasks were checked this way (printed under -s)."""
    from oracle.pyoracle import loop
    idx = np.flatnonzero((r.status != 4) & (o.status == 4))
    if idx.size:
        want = loop.run_task_loop([batch.task(int(i)) for i in idx], [batch.task_ids[int(i)].tobytes() for i in idx],
                                  o.handler, http_body=http)
        code = {"COMPLETE": 0, "ERROR": 1, "RETRY": 2, "REJECTED": 3}
        for i, w in zip(idx, want):
            assert (int(r.status[i]), r.result(int(i))) == (code[w.status], w.result), (int(i), batch.task(int(i))[:200])
        print(f"{o.handler}: {idx.size} task(s) the C oracle declines checked against the Python oracle")
    return int(idx.size)


def assert_matches_oracle(batch, r, o, allow_unsupported=0):
    """r: DrainResult from the device; o: coracle.OracleResult. Every task must agree exactly
    unless the device declared it UNSUPPORTED (then it must not have produced bytes). Where the C
    oracle declines and the device decided, the Python oracle decides. Returns that count."""
    assert r.n == batch.n
    assert np.array_equal(r.task_ids, batch.task_ids)
    unsup = r.status == 4
    assert int(unsup.sum()) <= allow_unsupported, f"{int(unsup.sum())} tasks UNSUPPORTED on the device"
    assert not np.any(r.has_result[unsup])
    ok = ~unsup & (o.status != 4)
    assert np.array_equal(r.status[ok], o.status[ok]), np.flatnonzero(ok & (r.status != o.status))[:10]
    assert np.array_equal(r.has_result[ok], o.has[ok])
    rl = r.lengths.astype(np.int64)
    ol = np.diff(o.offsets).astype(np.int64)
    assert np.array_equal(rl[ok], ol[ok]), np.flatnonzero(ok & (rl != ol))[:10]
    # every record lies inside the blob and records do not overlap (the blob may hold small gaps: slots
    # reserved for tasks that produced fewer bytes than the canonical frame predicts)
    assert int(rl.sum()) <= r.payload.size
    nz = np.flatnonzero(rl > 0)
    if nz.size:
        starts = r.offsets[nz].astype(np.int64); lens = rl[nz]
        order = np.argsort(starts, kind="stable")
        ends = starts[order] + lens[order]
        assert int(ends.max()) <= r.payload.size and np.all(ends[:-1] <= starts[order][1:])
    if not unsup.any() and not (o.status == 4).any():
        assert np.array_equal(r.fifo_payload(), o.payload)      # bit-for-bit, every record
    else:
        for i in np.flatnonzero(ok):
            assert r.result(i) == o.result(i), i
    return assert_matches_python_oracle_where_c_declines(batch, r, o)


def test_golden_fixtures(dq):
    g = G.load()
    for handler in HANDLERS:
        for name, cases in g["groups"].items():
            b = G.group_batch(cases)
            r = run_gpu(dq, b, handler)
            assert r.n == b.n
            for i, c in enumerate(cases):
                st, out = G.expected(c, handler)
                if r.status[i] == 4:
                    assert r.result(i) is None
                    continue
                assert (int(r.status[i]), r.result(i)) == (st, out), (name, i, c["payload"])


def test_identity_echo_10k_x_64(dq):
    b = synth.strings_batch(10_000, 64)           # BASELINE configs[0]
    r = run_gpu(dq, b, "identity")
    assert_matches_oracle(b, r, coracle.run_batch(b.task_ids, b.payload, b.offsets, "identity", nthreads=8))


def test_identity_adversarial_heavy(dq):
    b = synth.strings_batch(20_000, 256, adversarial_frac=0.5, seed=11)
    r = run_gpu(dq, b, "identity")
    assert_matches_oracle(b, r, coracle.run_batch(b.task_ids, b.payload, b.offsets, "identity", nthreads=8))


def test_identity_escaped_bodies_cooperative_check(dq):
    """The warp-cooperative canonical-escape check of the identity main loop (esc_verify_canonical): what json.dumps wrote,
    and mutations of it (raw quotes, "\\/", upper-case hex, lone / paired surrogates, odd backslash runs, raw non-ASCII,
    truncated escapes), at body lengths around the 16-byte lane chunks and the 512-byte passes."""
    import json
    import random
    from tests.test_esc_verify_model import MUT, rand_string
    rng = random.Random(77)
    payloads = []
    for k in range(24_000):
        n = rng.choice([1, 2, 7, 15, 16, 17, 31, 40, 100, 256, 300, 511, 512, 513, 700, 1500])
        body = bytearray(json.dumps(rand_string(rng, n, rng.random() < 0.4)).encode()[1:-1])
        if k % 3:
            for _ in range(rng.randint(1, 3)):
                pos = rng.randint(0, len(body))
                if rng.random() < 0.3 and len(body):
                    del body[pos:pos + rng.randint(1, 3)]
                else:
                    body[pos:pos] = rng.choice(MUT)
        payloads.append(b'{"args": ["' + bytes(body) + b'"], "kwargs": {}}')
    b = synth.from_payloads(payloads)
    r = run_gpu(dq, b, "identity")
    assert_matches_oracle(b, r, coracle.run_batch(b.task_ids, b.payload, b.offsets, "identity", nthreads=8))


def test_identity_1m_x_256_full_size(dq):
    b = synth.strings_batch(1_000_000, 256)       # BASELINE configs[1]
    r = run_gpu(dq, b, "identity")
    assert_matches_oracle(b, r, coracle.run_batch(b.task_ids, b.payload, b.offsets, "identity", nthreads=16))
    # size-independent property: draining the results of identity as strings again is idempotent
    assert int(r.status.sum()) == 0 and int(r.has_result.sum()) == b.n


def test_identity_on_other_configs(dq):
    for b in (synth.crc_batch(20_000), synth.vadd_batch(5000), synth.json_batch(300)):
        r = run_gpu(dq, b, "identity")
        o = coracle.run_batch(b.task_ids, b.payload, b.offsets, "identity", nthreads=8)
        assert_matches_oracle(b, r, o, allow_unsupported=b.n if b.name == "json_sum" else 0)


@pytest.mark.parametrize("handler", HANDLERS)
def test_handcrafted_edge_cases(dq, handler):
    from tests.test_oracle_c_vs_py import HANDCRAFTED
    b = synth.from_payloads(HANDCRAFTED)
    r = run_gpu(dq, b, handler)
    o = coracle.run_batch(b.task_ids, b.payload, b.offsets, handler)
    assert_matches_oracle(b, r, o, allow_unsupported=len(HANDCRAFTED))
    # the device may decline (UNSUPPORTED) only valid payloads whose arg is a float / non-empty container
    for i in np.flatnonzero(r.status == 4):
        # ... or a number with an exponent, whose float64 overflow (-> Ok:false) the device does not decide
        assert o.status[i] in (0, 4) or (o.status[i] == 3 and b"e" in HANDCRAFTED[i].lower()), HANDCRAFTED[i]


def test_crc32_zipf(dq):
    b = synth.crc_batch(50_000)                   # BASELINE configs[2] at a size the oracle does in seconds
    r = run_gpu(dq, b, "crc32")
    assert_matches_oracle(b, r, coracle.run_batch(b.task_ids, b.payload, b.offsets, "crc32", nthreads=16))
    b = synth.strings_batch(20_000, 256, adversarial_frac=0.3, seed=5)     # non-ASCII / escapes under the CRC
    r = run_gpu(dq, b, "crc32")
    assert_matches_oracle(b, r, coracle.run_batch(b.task_ids, b.payload, b.offsets, "crc32", nthreads=16))


def test_vadd_f32(dq):
    b = synth.vadd_batch(100_000)                 # BASELINE configs[3] payload shape
    r = run_gpu(dq, b, "vadd_f32")
    o = coracle.run_batch(b.task_ids, b.payload, b.offsets, "vadd_f32", nthreads=16)
    assert_matches_oracle(b, r, o)
    # float handler bodies within 1e-6 rel (north_star); here they are bit-equal, check the decoded values too
    import base64
    for i in (0, 1, b.n - 1):
        got = np.frombuffer(base64.b64decode(r.result(i)[1:-1]), "<f4")
        want = np.frombuffer(base64.b64decode(o.result(i)[1:-1]), "<f4")
        assert np.allclose(got, want, rtol=1e-6, atol=0)
    for fpv in list(range(1, 14)) + [31, 33, 64, 100]:      # every base64 phase of a, of b and of the padding
        b = synth.vadd_batch(300, floats_per_vec=fpv, seed=fpv)
        r = run_gpu(dq, b, "vadd_f32")
        assert_matches_oracle(b, r, coracle.run_batch(b.task_ids, b.payload, b.offsets, "vadd_f32"))
        b = synth.vadd_special_batch(300, floats_per_vec=fpv, seed=fpv)     # NaN payloads, inf - inf, denormals
        r = run_gpu(dq, b, "vadd_f32")
        assert_matches_oracle(b, r, coracle.run_batch(b.task_ids, b.payload, b.offsets, "vadd_f32"))


def test_vadd_f32_corrupted_text(dq):
    """One wrong character anywhere in an otherwise canonical task (outside the alphabet, '=' in the
    middle, a missing character, an odd float count) must come out exactly as the oracle says."""
    rng = np.random.default_rng(77)
    payloads = []
    for fpv in (1, 2, 3, 4, 32):
        base = synth.vadd_batch(40, floats_per_vec=fpv, seed=100 + fpv)
        for i in range(base.n):
            p = bytearray(base.payload[int(base.offsets[i]):int(base.offsets[i + 1])].tobytes())
            lo, hi = 11, len(p) - 17
            kind = i % 5
            pos = int(rng.integers(lo, hi))
            if kind == 0: p[pos] = rng.choice(list(b"!#$%&'()*,-.:;<>?@[]^_`{|}~ \x7f\"\\\n"))
            elif kind == 1: p[pos] = ord("=")
            elif kind == 2: del p[pos]
            elif kind == 3: p[pos:pos] = b"AAAA"           # four more characters: three more bytes, not two vectors any more
            else: p[pos] = 0xC3                            # not ASCII (and not valid UTF-8)
            payloads.append(bytes(p))
    b = synth.from_payloads(payloads)
    r = run_gpu(dq, b, "vadd_f32")
    assert_matches_oracle(b, r, coracle.run_batch(b.task_ids, b.payload, b.offsets, "vadd_f32"))


def test_json_sum(dq):
    b = synth.json_batch(20_000)                  # BASELINE configs[4] payload shape
    r = run_gpu(dq, b, "json_sum")
    assert_matches_oracle(b, r, coracle.run_batch(b.task_ids, b.payload, b.offsets, "json_sum", nthreads=16))


def test_json_sum_fast_path_boundaries_and_mutants(dq):
    """The warp-cooperative parser: numbers straddling every 32-byte lane boundary, documents around
    the 1 KiB limit, both separator styles, and single-character mutants of canonical documents."""
    import json
    from tests.test_json_coop_model import _large_payloads, _payloads
    rng = np.random.default_rng(0xB9 + 7)
    payloads = _payloads(rng, 800) + _large_payloads(rng, 400)
    for shift in range(0, 70):                     # slide a run of 15-digit and short numbers across the lane boundaries
        d = {"p": "x" * shift, "values": [999999999999999, 7, 123456789012345, 0, 10, 100000000000000] * 3, "q": 5}
        payloads.append(json.dumps({"args": [d], "kwargs": {}}).encode())
    for shift in range(940, 1080, 3):              # ... and across the 1 KiB segment boundary of longer documents
        d = {"p": "x" * shift, "values": [999999999999999, 7, 123456789012345, 0, 10, 100000000000000] * 3, "q": "]", "values2": [1]}
        payloads.append(json.dumps({"args": [d], "kwargs": {}}).encode())
    n_canonical = 70 + len(range(940, 1080, 3)) + 14
    for size in (900, 1000, 1023, 1024, 1025, 1100, 2047, 2048, 2049, 3000, 4095, 4096, 4097, 5000):      # around the segment and JSON_COOP_MAX_DOC limits
        vals = rng.integers(0, 10**6, size=60).tolist()
        d = {"id": size, "values": vals, "pad": ""}
        d["pad"] = "y" * max(0, size - len(json.dumps(d)))
        payloads.append(json.dumps({"args": [d], "kwargs": {}}).encode())
    b = synth.from_payloads(payloads)
    r = run_gpu(dq, b, "json_sum")
    o = coracle.run_batch(b.task_ids, b.payload, b.offsets, "json_sum", nthreads=16)
    assert_matches_oracle(b, r, o, allow_unsupported=b.n)
    for i in np.flatnonzero(r.status == 4):        # declined only where the oracle's domain ends too, or on exotic numbers
        assert o.status[i] in (0, 3, 4), payloads[i]
    # the canonical documents must not be declined
    assert int((r.status[-n_canonical:] == 4).sum()) == 0


def test_async_launch_then_fetch(dq):
    """B9_DRAIN_ASYNC: launches return at once; sync / fetch publish the same records a blocking launch gives."""
    b = synth.strings_batch(50_000, 64, adversarial_frac=0.05, seed=9)
    o = coracle.run_batch(b.task_ids, b.payload, b.offsets, "identity", nthreads=8)
    dq.push_batch(b.task_ids, b.payload, b.offsets)
    for _ in range(3):                                           # back to back on the same resident window
        assert dq.drain_launch("identity", b.n, peek=True, wait=False) == b.n
    dq.sync()
    assert dq.depth() == b.n                                     # peeked: still pending
    assert dq.drain_launch("identity", b.n, peek=False, wait=False) == b.n
    r = dq.fetch()                                               # completes the launch, then pops
    assert dq.depth() == 0 and r.n_popped == b.n
    assert_matches_oracle(b, r, o)


def _http_bodies():
    """HTTP request bodies for B9_TF_HTTP_BODY: the reference's own SerializeHttpPayload cases
    (pkg/task/serialize_test.go:39-173, those without a query string), map-rule corner cases, SDK-framed
    payloads (valid bodies too), and single-character mutants."""
    import json
    from tests.test_oracle_reference_answers import SERIALIZE_CASES
    bodies = [c[1].encode() for c in SERIALIZE_CASES if not c[2]]
    bodies += [b'{"args": ["abc"]}', b'{"args": ["abc"], "kwargs": {}}', b'{"x": 1}', b'', b'  \n', b'null', b'[1]', b'"s"', b'7',
               b'{"args": "notalist"}', b'{"args": null}', b'{"args": ["a"], "kwargs": 5}', b'{"args": ["a"], "kwargs": null}',
               b'{"args": ["a"], "other": [1e999]}', b'{"args": ["a"], "other": 1e400, "kwargs": {}}', b'{"\\u0061rgs": ["esc"]}',
               b'{"Args": ["folded?"]}', b'{"ARGS": ["x"], "KWARGS": {}}', b'{"args": ["a"], "args": 1}', b'{"args": 1, "args": ["last"]}',
               b'{"args": ["x"], "kwargs": {"a": 1}}', b' {"args":["ws"]} ', b'{"kwargs": {}, "args": ["order"]}', b'{"kwargs": {"k": 1}, "kwargs": {}, "args": ["dup kw"]}',
               b'{"kwargs": {}, "kwargs": {"k": 1}, "args": ["dup kw 2"]}', b'{"args": ["x"], "kwargs": {}, "extra": true}', b'{"args": ["x"], "extra": true}',
               b'{"args": []}', b'{"args": ["a", "b"]}', b'{"args": [""]}', b'{"args": [0]}', b'{"args": [123]}', b'{"args": [{"values": [1, 2, 3]}]}',
               b'{"args": [{"values": [1, 2, 3]}], "kwargs": {}}', b'{"args": ["QUJDRA=="]}', b'{"args": ["AACAPwAAgD8="]}', b'{}', b'{"args": ["x"]} trailing',
               b'{"args": ["\\ud83d\\ude00 \\u00e9"]}', b'{"args": ["a\\/b"]}', b'{"k\\u0077args": {}, "args": ["esc key"]}']
    rng = np.random.default_rng(4242)
    sdk = synth.strings_batch(60, 40, adversarial_frac=0.3, seed=77)
    bodies += [sdk.task(i) for i in range(sdk.n)]
    jb = synth.json_batch(6, doc_bytes=300)
    bodies += [jb.task(i) for i in range(jb.n)]
    vb = synth.vadd_batch(6, floats_per_vec=4)
    bodies += [vb.task(i) for i in range(vb.n)]
    base = list(bodies)
    alphabet = list(b'{}[],:" 01e.-nulltrackwgs\\')
    for b in base:
        if len(b) < 4:
            continue
        for _ in range(3):
            m = bytearray(b)
            pos = int(rng.integers(0, len(m)))
            op = int(rng.integers(0, 3))
            ch = int(rng.choice(alphabet))
            if op == 0: m[pos] = ch
            elif op == 1: del m[pos]
            else: m[pos:pos] = bytes([ch])
            bodies.append(bytes(m))
    return bodies


@pytest.mark.parametrize("handler", HANDLERS)
def test_http_body_mode(dq, handler):
    """B9_TF_HTTP_BODY: args / kwargs by SerializeHttpPayload's map rules, against the Python oracle
    (its serialize_http_payload is pinned to the reference's 15 known answers)."""
    from oracle.pyoracle import loop
    bodies = _http_bodies()
    b = synth.from_payloads(bodies)
    assert dq.depth() == 0
    dq.push_batch(b.task_ids, b.payload, b.offsets, flags=np.full(b.n, 2, np.uint8))
    r = dq.drain(handler, max_tasks=b.n)
    assert r.n == b.n and dq.depth() == 0
    want = loop.run_task_loop(bodies, [bytes(x) for x in b.task_ids], handler, http_body=True)
    code = {"COMPLETE": 0, "ERROR": 1, "RETRY": 2, "REJECTED": 3}
    declined = 0
    for i, w in enumerate(want):
        if r.status[i] == 4:                       # floats etc.: the device declines, never guesses
            assert not r.has_result[i]
            assert w.status in ("COMPLETE", "ERROR", "REJECTED"), bodies[i]
            declined += 1
            continue
        assert r.status[i] == code[w.status], (bodies[i], int(r.status[i]), w.status)
        assert r.result(i) == w.result, (bodies[i], r.result(i), w.result)
    assert declined <= len(bodies) // 10
    # the same bytes WITHOUT the flag follow the struct rules: e.g. an empty body is refused, unknown keys are ignored
    plain = [b'', b'{"args": ["x"], "extra": true}', b'{"Args": ["folded"]}']
    pb = synth.from_payloads(plain)
    dq.push_batch(pb.task_ids, pb.payload, pb.offsets)
    r2 = dq.drain("identity", max_tasks=pb.n)
    assert list(r2.status) == [3, 0, 0] and r2.result(1) == b'"x"' and r2.result(2) == b'"folded"'


def test_wrong_handler_for_payload(dq):
    # every handler over every config's payloads: type errors must come out as ERROR exactly like the oracle
    for b in (synth.strings_batch(2000, 64, adversarial_frac=0.2), synth.vadd_batch(1000), synth.json_batch(200)):
        for h in HANDLERS:
            r = run_gpu(dq, b, h)
            o = coracle.run_batch(b.task_ids, b.payload, b.offsets, h)
            assert_matches_oracle(b, r, o, allow_unsupported=b.n if (h == "identity" and b.name == "json_sum") else 0)


def test_empty_and_ragged(dq):
    assert dq.drain("identity").n == 0                      # empty queue
    payloads = [b"", b"{}", b'{"args": [""], "kwargs": {}}', b'{"args": ["' + b"x" * 70000 + b'"], "kwargs": {}}',
                b'{"args": ["a"], "kwargs": {}}']
    b = synth.from_payloads(payloads)
    r = run_gpu(dq, b, "identity")
    assert_matches_oracle(b, r, coracle.run_batch(b.task_ids, b.payload, b.offsets, "identity"))


def test_fifo_across_pushes_partial_drains_and_wrap():
    from beta9_b200.device_queue import DeviceQueue
    from beta9_b200 import _lib as L
    q = DeviceQueue(ring_bytes=1 << 20, ring_tasks=1 << 12, max_drain_tasks=1 << 12, max_result_bytes=1 << 21)
    try:
        rng = np.random.default_rng(5)
        pending = []          # (task_id bytes, expected result)
        seed = 100
        for step in range(60):
            n = int(rng.integers(1, 700))
            b = synth.strings_batch(n, int(rng.integers(1, 300)), adversarial_frac=0.1, seed=seed)
            seed += 1
            try:
                q.push_batch(b.task_ids, b.payload, b.offsets)
            except L.B9Error as e:
                assert e.code == L.B9_ENOSPC          # ring full: nothing appended
                b = None
            if b is not None:
                o = coracle.run_batch(b.task_ids, b.payload, b.offsets, "identity")
                pending += [(b.task_ids[i].tobytes(), int(o.status[i]), o.result(i)) for i in range(b.n)]
            assert q.depth() == len(pending)
            take = int(rng.integers(0, 900))
            r = q.drain("identity", max_tasks=take)
            assert r.n == min(take, len(pending))
            for i in range(r.n):
                tid, st, res = pending[i]
                assert r.task_ids[i].tobytes() == tid and int(r.status[i]) == st and r.result(i) == res
            pending = pending[r.n:]
        r = q.drain("identity")
        assert r.n == len(pending)
        assert q.depth() == 0 and q.depth_bytes() == 0
    finally:
        q.close()


def test_cancelled_and_expired_tasks_are_compacted_away(dq):
    b = synth.strings_batch(5000, 64, seed=21)
    rng = np.random.default_rng(3)
    flags = (rng.random(b.n) < 0.3).astype(np.uint8)               # B9_TF_CANCELLED
    expires = np.where(rng.random(b.n) < 0.2, 1_000, 0).astype(np.int64)   # already expired
    expires[rng.random(b.n) < 0.2] = 10**19 // 2                     # far future
    dq.push_batch(b.task_ids, b.payload, b.offsets, expires_unix_ns=expires, flags=flags)
    n_exp = dq.expire(now_unix_ns=2_000)
    gone = (flags != 0) | (expires == 1_000)
    assert n_exp == int(((expires == 1_000) & (flags == 0)).sum())
    r = dq.drain("identity")
    assert r.n_popped == b.n and r.n == int((~gone).sum())
    o = coracle.run_batch(b.task_ids, b.payload, b.offsets, "identity")
    keep = np.flatnonzero(~gone)
    assert np.array_equal(r.task_ids, b.task_ids[keep])
    for j, i in enumerate(keep):
        assert int(r.status[j]) == int(o.status[i]) and r.result(j) == o.result(i)


@pytest.mark.parametrize("handler,make", [("identity", lambda: synth.strings_batch(70_001, 48, adversarial_frac=0.02, seed=31)),
                                          ("crc32", lambda: synth.crc_batch(3001, seed=32)),
                                          ("vadd_f32", lambda: synth.vadd_batch(9007, seed=33)),
                                          ("json_sum", lambda: synth.json_batch(1203, doc_bytes=400, seed=34))])
def test_cancelled_slots_every_handler(dq, handler, make):
    """Record indices with cancelled slots in the window (tile_count_kernel / tile_scan_kernel ahead of the drain),
    for every warp-tile size (32, 4 and 8 slots), odd task counts, runs of cancelled slots, a single one, all but one."""
    b = make()
    o = coracle.run_batch(b.task_ids, b.payload, b.offsets, handler, nthreads=8)
    rng = np.random.default_rng(b.n)
    patterns = [rng.random(b.n) < 0.07, np.arange(b.n) == b.n // 3, np.arange(b.n) != 5,
                (np.arange(b.n) // 97) % 3 == 0, np.arange(b.n) < 40, np.arange(b.n) >= b.n - 33]
    for gone in patterns:
        dq.push_batch(b.task_ids, b.payload, b.offsets, flags=gone.astype(np.uint8))
        r = dq.drain(handler)
        keep = np.flatnonzero(~gone)
        assert r.n_popped == b.n and r.n == keep.size and dq.depth() == 0
        assert np.array_equal(r.task_ids, b.task_ids[keep])
        assert np.array_equal(r.status, o.status[keep]) and np.array_equal(r.has_result, o.has[keep])
        for j in list(range(min(50, keep.size))) + list(range(max(0, keep.size - 50), keep.size)) + list(rng.integers(0, keep.size, 200)):
            assert r.result(int(j)) == o.result(int(keep[int(j)])), (handler, int(j))


def test_result_capacity_errors_do_not_consume():
    from beta9_b200.device_queue import DeviceQueue
    from beta9_b200 import _lib as L
    q = DeviceQueue(ring_bytes=1 << 22, ring_tasks=1 << 12, max_drain_tasks=1 << 12, max_result_bytes=1 << 12)
    try:
        b = synth.strings_batch(1000, 64, adversarial_frac=0)
        q.push_batch(b.task_ids, b.payload, b.offsets)
        with pytest.raises(L.B9Error) as e:
            q.drain("identity")
        assert e.value.code == L.B9_ENOSPC and q.depth() == 1000       # staging too small: nothing consumed
        r = q.drain("identity", max_tasks=50)                            # 50 x 66 B fits
        assert r.n == 50 and q.depth() == 950
        with pytest.raises(L.B9Error) as e:
            q.push_batch(b.task_ids[:1], np.zeros(3 << 20, np.uint8), np.array([0, 3 << 20], np.uint64))
        assert e.value.code in (L.B9_E2BIG, L.B9_EINVAL)
    finally:
        q.close()


# ---- BASELINE.json configs at their stated per-GPU sizes (VERDICT r1: parity was run at reduced sizes for 3 of 4 configs)
def test_crc32_1m_zipf_full_size():
    """configs[2]: 1M zipf 32..4096-char strings through crc32, every record against the oracle."""
    from beta9_b200.device_queue import DeviceQueue
    b = synth.crc_batch(1_000_000)
    with DeviceQueue(ring_bytes=2 << 30, ring_tasks=1 << 21, max_drain_tasks=1 << 21, max_result_bytes=1 << 28) as q:
        r = run_gpu(q, b, "crc32")
    o = coracle.run_batch(b.task_ids, b.payload, b.offsets, "crc32", nthreads=32, out_cap=16 * b.n + 64)
    assert_matches_oracle(b, r, o)
    assert int(r.status.sum()) == 0


def test_json_sum_100k_full_size(dq):
    """configs[4]: 100k x 1 KB JSON documents through json_sum."""
    b = synth.json_batch(100_000)
    r = run_gpu(dq, b, "json_sum")
    assert_matches_oracle(b, r, coracle.run_batch(b.task_ids, b.payload, b.offsets, "json_sum", nthreads=32, out_cap=24 * b.n + 64))
    assert int(r.status.sum()) == 0 and int(r.has_result.sum()) == b.n


def test_vadd_f32_per_gpu_share_of_10m(dq):
    """configs[3]: 10M x 256 B fp32 vector-add over 8 GPUs = 1.25M tasks per GPU; float results within 1e-6 rel
    (north_star) — they are bit-equal to the oracle's (numpy's IEEE add), which is stricter."""
    b = synth.vadd_batch(1_250_000)
    r = run_gpu(dq, b, "vadd_f32")
    o = coracle.run_batch(b.task_ids, b.payload, b.offsets, "vadd_f32", nthreads=32, out_cap=200 * b.n + 64)
    assert_matches_oracle(b, r, o)
    import base64
    for i in range(0, b.n, 100_003):
        got = np.frombuffer(base64.b64decode(r.result(i)[1:-1]), "<f4")
        want = np.frombuffer(base64.b64decode(o.result(i)[1:-1]), "<f4")
        assert np.allclose(got, want, rtol=1e-6, atol=0)
