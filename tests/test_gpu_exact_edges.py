"""GPU: json_sum and crc32 at their exact edges, and crc32 / identity with one unit of every kind placed around every
lane's chunk boundary, against the Python oracle's task loop (exact everywhere): status and result bytes equal, or, for
json_sum only, a decline (UNSUPPORTED, no bytes) where a partial sum leaves int64.

Paths covered: json_sum's warp-cooperative parser (canonical documents <= 4 KiB of non-negative <= 15-digit values) and
its sequential one (longer documents, negative values, true / false, HTTP bodies); crc32's warp-cooperative scan over
staged bodies (shared memory) and unstaged ones (tasks larger than the stage buffer, up to 1 MiB), with bodies long
enough to use every level of the zero-byte shift; the sequential crc32 and the identity tail's chunked transcoder."""
import json
import random

import numpy as np
import pytest

from beta9_b200 import synth
from oracle.pyoracle import loop
from tests.test_exact_edges_on_host import (CODE, DETOUR_AT, crc_targets, filler, forced_string, plain_values,
                                            sum_answer_error, sum_lists, sum_targets)

pytestmark = pytest.mark.gpu

MAX_TASK = 1 << 20                      # DeviceQueue's default max_task_bytes


@pytest.fixture(scope="module")
def dq():
    from beta9_b200.device_queue import DeviceQueue
    q = DeviceQueue(ring_bytes=1 << 31, ring_tasks=1 << 20, max_drain_tasks=1 << 20, max_result_bytes=1 << 31)
    yield q
    q.close()


def drain(dq, payloads, handler, http=False):
    b = synth.from_payloads(payloads)
    assert dq.depth() == 0
    if http:
        dq.push_batch(b.task_ids, b.payload, b.offsets, flags=np.full(b.n, 2, np.uint8))
    else:
        dq.push_batch(b.task_ids, b.payload, b.offsets)
    r = dq.drain(handler, max_tasks=b.n)
    assert r.n == b.n and dq.depth() == 0 and np.array_equal(r.task_ids, b.task_ids)
    return b, r


def assert_exact(dq, payloads, handler):
    """Every task's status and bytes are the Python oracle's (no declines: strings are always decided)."""
    b, r = drain(dq, payloads, handler)
    want = loop.run_task_loop(payloads, [bytes(x) for x in b.task_ids], handler)
    bad = [(i, int(r.status[i]), r.result(i) if r.result(i) is None else r.result(i)[:60], w.status,
            w.result if w.result is None else w.result[:60], payloads[i][:120])
           for i, w in enumerate(want) if (int(r.status[i]), r.result(i)) != (CODE[w.status], w.result)]
    assert not bad, f"{len(bad)} of {len(payloads)} wrong:\n" + "\n".join(map(str, bad[:20]))


# ---------------------------------------------------------------- json_sum
def test_json_sum_exact_edges_both_paths(dq):
    cases = []                                                            # (payload, values, http)
    for t in sum_targets():
        if 0 <= t:                                                        # canonical documents: the cooperative parser
            vals = plain_values(t)
            for doc in (json.dumps({"values": vals}), json.dumps({"id": 7, "values": vals}, separators=(",", ":"))):
                if len(doc) <= 4096:
                    cases.append((b'{"args": [' + doc.encode() + b'], "kwargs": {}}', vals, False))
        for name, vals in sum_lists(t, detour=abs(t) in DETOUR_AT):       # the sequential parser
            p = loop.sdk_put_payload({"values": vals, "pad": "p" * 4200})   # (> 4 KiB even when the list is short)
            if len(p) <= MAX_TASK:
                cases.append((p, vals, False))
    for t in (1, -1, 2**32 + 1, -(2**32) - 1, 4294967296 * 10**9 + 1, 2**62, 2**63 - 1, -2**63, 2**63):
        vals = plain_values(t)
        cases.append((b'{"args": [' + json.dumps({"values": vals}).encode() + b"]}", vals, True))
    n_coop = sum(1 for p, _, h in cases if not h and len(p) <= 4096 + 30)
    assert n_coop >= 40
    bad, declined = [], 0
    for http in (False, True):
        sel = [c for c in cases if c[2] == http]
        b, r = drain(dq, [p for p, _, _ in sel], "json_sum", http=http)
        for i, (p, vals, _) in enumerate(sel):
            st, res = int(r.status[i]), r.result(i)
            declined += st == 4
            err = sum_answer_error(p, vals, st, res, http=http)
            if err:
                bad.append((sum(vals), len(p), http) + err)
    assert not bad, "\n".join(map(str, bad))
    assert declined >= 16


# ---------------------------------------------------------------- crc32, forced values
def test_crc32_forced_values_staged_and_unstaged(dq):
    """Bodies of ~30 B, ~300 B and ~20 KB fit the stage buffer (<= 48 KiB per warp); ~200 KB and ~1 MiB do not and are
    read from global memory. The same strings in another frame take the sequential parser."""
    strings = []
    for n in (30, 300, 20_000, 200_000, 900_000):
        targets = crc_targets() if n <= 200_000 else [0, 1, 9, 10**9, 2**31, 2**32 - 1]
        for t in targets:
            strings.append(forced_string(filler(n, seed=n + t % 1009), t))
    payloads = [loop.sdk_put_payload(s) for s in strings]
    assert max(map(len, payloads)) <= MAX_TASK
    payloads += [b'{"args":[' + json.dumps(s).encode() + b'],"kwargs":{}}' for s in strings[::3]]
    assert_exact(dq, payloads, "crc32")


def test_crc32_long_bodies(dq):
    """Unforced bodies from 2^13 to ~2^20 bytes, escaped (json.dumps) and raw UTF-8, so that the zero-byte shift uses
    its upper levels; and the same through identity."""
    payloads = []
    for n in (8_200, 16_400, 40_000, 70_000, 131_100, 300_000, 600_000, 900_000):
        s = filler(n, seed=n)
        payloads.append(loop.sdk_put_payload(s))
        raw = json.dumps({"args": [s], "kwargs": {}}, ensure_ascii=False).encode()
        if len(raw) <= MAX_TASK:
            payloads.append(raw)
    assert_exact(dq, payloads, "crc32")
    assert_exact(dq, payloads, "identity")


# ---------------------------------------------------------------- units at chunk boundaries
UNITS = (["é".encode(), "€".encode(), "😀".encode()]                                                 # valid raw UTF-8
         + [b"\x80", b"\xc3", b"\xe2\x82", b"\xf0\x9f\x98", b"\xc0\x80", b"\xed\xa0\x80", b"\xf5"]  # invalid UTF-8
         + [b"\\u00e9", b"\\u00E9", b"\\u20ac", b"\\u20AC", b"\\uabcd"]                                 # \uXXXX
         + [b"\\ud83d", b"\\uDE00", b"\\ud83d\\ude00", b"\\uD83D\\uDE00", b"\\ude00\\ud83d"]             # surrogates
         + [b"\\/", b"\\b", b"\\f", b"\\n", b"\\r", b"\\t", b'\\"', b"\\\\"]
         + [b"\\" * k + b"u" for k in range(2, 10)])                                                   # backslash runs + u
LENGTHS = list(range(1, 41)) + [63, 64, 65, 95, 96, 97, 255, 256, 257, 1000, 4097, 20000]
FILL = b"x0y1z2Aa3Bb4Cc5Dd6Ee7Ff8 9-"                   # plain ASCII; hex digits among it complete some \u runs


def boundary_payloads():
    """One unit at l * ceil(n/32) + d, d = -12..+6, for a spread of lanes l (all of them for n <= 40, fewer for the long
    bodies), clipped into the body; the rest of the body is FILL from an offset that varies with (n, unit)."""
    out = set()
    for n in LENGTHS:
        S = -(-n // 32)
        spread = range(1, 32) if n <= 40 else (1, 2, 7, 15, 16, 17, 30, 31) if n <= 257 else (1, 15, 16, 31) if n <= 1000 else \
            (1, 16, 31) if n <= 4097 else (16,)
        for j, u in enumerate(UNITS):
            if len(u) > n:
                continue
            k = (7 * n + 5 * j) % len(FILL)
            fill = (FILL * (n // len(FILL) + 2))[k:k + n]
            for l in spread:
                for d in range(-12, 7):
                    pos = min(max(l * S + d, 0), n - len(u))
                    out.add(synth.PREFIX + fill[:pos] + u + fill[pos + len(u):] + synth.SUFFIX)
    out = sorted(out)
    random.Random(32).shuffle(out)
    return out


@pytest.mark.parametrize("handler", ["crc32", "identity"])
def test_units_at_chunk_boundaries(dq, handler):
    payloads = boundary_payloads()
    assert 10_000 <= len(payloads) <= 80_000
    assert_exact(dq, payloads, handler)
