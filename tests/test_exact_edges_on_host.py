"""The device's sequential json_sum and crc32 (handler_seq.cuh, compiled for the host by tests/host_shim/host_parse.cpp)
at the values where integer code goes wrong, against the Python oracle: json_sum totals at every change of decimal
length up to 10^20, at the 32-bit limb switches of the decimal writer and at the int64 / uint64 limits, in both signs;
crc32 results forced to 0, to small numbers, to every power of ten and to 2^31 and 2^32 - 1 by four appended characters.

The generators here are shared with tests/test_gpu_exact_edges.py, which puts the same values through the kernels."""
import json
import zlib

import pytest

from oracle.pyoracle import loop
from tests.test_device_parser_on_host import load_host_shim

INT64_MIN, INT64_MAX = -2**63, 2**63 - 1
BIG = 10**15 - 1                      # the largest magnitude the device sums as an integer (<= 15 digits)
CODE = {"COMPLETE": 0, "ERROR": 1, "RETRY": 2, "REJECTED": 3}
JSON_SUM, CRC32 = 3, 1                # handler numbers of b9_host_run


@pytest.fixture(scope="module")
def shim():
    return load_host_shim()


# ---------------------------------------------------------------- json_sum
def sum_targets():
    """10^k - 1, 10^k, 10^k + 1 for k = 0..20; 2^32 and 4294967296 * 10^9 (where write_dec goes from one 9-digit limb
    to two, and from two to three) and 2^62, each +-1; 2^63 - 1, 2^63, 2^64 - 1, 2^64. Both signs."""
    t = set()
    for k in range(21):
        t |= {10**k - 1, 10**k, 10**k + 1}
    for c in (2**32, 4294967296 * 10**9, 2**62):
        t |= {c - 1, c, c + 1}
    t |= {INT64_MAX, 2**63, 2**64 - 1, 2**64}
    return sorted(t | {-x for x in t})


def plain_values(total):
    """<= 15-digit integers of one sign adding up to `total`: the partial sums run monotonically from 0 to it."""
    s = -1 if total < 0 else 1
    q, r = divmod(abs(total), BIG)
    return [s * BIG] * q + ([s * r] if r else [])


def sum_lists(total, detour=False):
    """(name, values) lists with sum(values) == total: plain; with true / false in front (True counts 1); and, with
    `detour`, lists whose partial sums leave int64 and come back, or touch its limit exactly and come back."""
    out = [("plain", plain_values(total)), ("bools", [True, False, True, True, False] + plain_values(total - 3))]
    if detour:
        e = INT64_MAX // BIG + 2                                          # e * BIG > 2^63: past the limit
        s = -1 if total < 0 else 1
        out.append(("out_and_back", [s * BIG] * e + [-s * BIG] * e + plain_values(total)))
        out.append(("to_max_and_back", plain_values(INT64_MAX) + plain_values(total - INT64_MAX)))
        out.append(("to_min_and_back", plain_values(INT64_MIN) + plain_values(total - INT64_MIN)))
    return out


def leaves_int64(values):
    p = 0
    for v in values:
        p += v
        if not INT64_MIN <= p <= INT64_MAX:
            return True
    return False


def sum_payload(values, pad=0):
    doc = {"values": values}
    if pad:
        doc["pad"] = "p" * pad
    return loop.sdk_put_payload(doc)


def sum_answer_error(payload, values, st, res, http=False):
    """None if the device's (status, bytes) are right, else what is wrong. Right is: what the Python oracle answers, or
    a decline (status 4, no bytes) — and that only where a partial sum of the list leaves int64, which is all that can
    make the device decline a list of <= 15-digit integers and booleans. (The oracle is only run where it is compared
    with: it takes seconds on the megabyte-sized documents the device declines.)"""
    if st == 4:
        return None if res is None and leaves_int64(values) else ("declined", st, res)
    w = loop.run_task_loop([payload], [bytes(16)], "json_sum", http_body=http)[0]
    return None if (st, res) == (CODE[w.status], w.result) else (st, res, w.status, w.result)


DETOUR_AT = {0, 1, 10**15, 2**62 + 1, INT64_MAX, 2**63}


def sum_cases():
    cases = []
    for t in sum_targets():
        for name, vals in sum_lists(t, detour=abs(t) in DETOUR_AT):
            assert sum(vals) == t
            cases.append((t, name, vals))
    return cases


def test_json_sum_exact_at_decimal_and_int64_edges(shim):
    bad, declined = [], 0
    cases = sum_cases()
    for t, name, vals in cases:
        p = sum_payload(vals)
        st, res = shim.run(p, False, JSON_SUM)
        declined += st == 4
        err = sum_answer_error(p, vals, st, res)
        if err:
            bad.append((t, name) + err)
    assert not bad, "\n".join(map(str, bad))
    assert len(cases) - declined > 250 and declined >= 16


def test_json_sum_int64_min_prints_like_python(shim):
    st, res = shim.run(sum_payload(plain_values(INT64_MIN)), False, JSON_SUM)
    assert (st, res) == (0, b"-9223372036854775808")
    st, res = shim.run(sum_payload([True] + plain_values(INT64_MAX - 1)), False, JSON_SUM)
    assert (st, res) == (0, b"9223372036854775807")
    st, res = shim.run(sum_payload(plain_values(INT64_MAX) + [True]), False, JSON_SUM)     # True takes it past the limit
    assert (st, res) == (4, None)


# ---------------------------------------------------------------- crc32
def forge4(prefix: bytes, target: int, start: int = 0):
    """Four bytes x with zlib.crc32(prefix + x, start) == target, or None. CRC-32 is affine in the message bits: solve
    the 32 x 32 system over GF(2) whose columns are the CRC changes of the 32 single-bit messages."""
    c = zlib.crc32(prefix + bytes(4), start)
    basis = {}                                                           # pivot bit -> (column combination, bits of x)
    for j in range(32):
        v, m = zlib.crc32(prefix + (1 << j).to_bytes(4, "little"), start) ^ c, 1 << j
        while v:
            h = v.bit_length() - 1
            if h not in basis:
                basis[h] = (v, m)
                break
            v, m = v ^ basis[h][0], m ^ basis[h][1]
    need, x = target ^ c, 0
    while need:
        h = need.bit_length() - 1
        if h not in basis:
            return None
        need, x = need ^ basis[h][0], x ^ basis[h][1]
    return x.to_bytes(4, "little")


def forced_string(prefix: str, target: int) -> str:
    """prefix + two more characters + four ASCII characters such that zlib.crc32(s.encode()) == target. The two extra
    characters are retried until all four forged bytes are ASCII (json.dumps escapes the controls and quotes among them)."""
    start = zlib.crc32(prefix.encode())
    for k in range(4096):
        head = chr(0x21 + k % 94) + chr(0x21 + k // 94 % 94)
        x = forge4(head.encode(), target, start)
        if x is not None and max(x) < 0x80:
            s = prefix + head + x.decode("ascii")
            assert zlib.crc32(s.encode()) == target
            return s
    raise AssertionError("no ASCII preimage found")


def crc_targets():
    return [0] + list(range(1, 11)) + [10**k - 1 for k in range(2, 10)] + [10**k for k in range(1, 10)] + [2**31, 2**32 - 1]


def filler(n: int, seed: int) -> str:
    """n characters of mostly printable ASCII with some that json.dumps escapes (quotes, backslashes, controls,
    non-ASCII, astral characters as surrogate pairs)."""
    import random
    rng = random.Random(seed)
    pool = [chr(c) for c in range(0x20, 0x7F)] * 4 + ['"', "\\", "\n", "\x01", "é", "€", "\U0001f600", "/"]
    return "".join(rng.choice(pool) for _ in range(n))


def test_crc32_forced_values(shim):
    strings = []
    for t in crc_targets():
        for n in (0, 1, 30, 300):
            strings.append((t, forced_string(filler(n, seed=n * 7 + t % 97), t)))
    payloads = [loop.sdk_put_payload(s) for _, s in strings]
    payloads += [b'{"args":[' + json.dumps(s).encode() + b"]}" for _, s in strings]     # another frame, same strings
    want = loop.run_task_loop(payloads, [bytes(16)] * len(payloads), "crc32")
    for (t, s), p, w in zip(strings * 2, payloads, want):
        st, res = shim.run(p, False, CRC32)
        assert w.status == "COMPLETE" and w.result == (str(t).encode() if t else None)
        assert (st, res) == (0, w.result), (t, s, st, res)
