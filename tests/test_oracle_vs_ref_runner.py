"""The oracle against the REFERENCE ITSELF: tests/golden/ref_runner_golden.json holds what the
reference's own runner loop (sdk/src/beta9/runner/taskqueue.py:297-404, imported unmodified by
tests/golden/make_ref_runner_golden.py) completed each golden wire record with, and what the
reference's own `_CallableWrapper.put` (sdk/src/beta9/abstractions/taskqueue.py:254-295) built for each
golden argument list. This pins rows a1 and a10-a12 of SURVEY.md §8 (put payload, json.loads ->
handler call convention -> falsy rule -> serialize_result -> task status) to the reference's code; the
Go half of the wire record stays a restatement."""
import base64
import json
import os

import pytest

from oracle.pyoracle import loop

HERE = os.path.dirname(os.path.abspath(__file__))
HANDLERS = ["identity", "crc32", "vadd_f32", "json_sum"]


@pytest.fixture(scope="module")
def goldens():
    hot = json.load(open(os.path.join(HERE, "golden", "hot_path_golden.json")))
    ref = json.load(open(os.path.join(HERE, "golden", "ref_runner_golden.json")))
    return hot, ref


def test_every_wire_record_went_through_the_reference_runner(goldens):
    hot, ref = goldens
    n = 0
    for g, cases in hot["groups"].items():
        for i, c in enumerate(cases):
            if c["wire"] is None:
                assert str(i) not in ref["groups"].get(g, {})          # refused at put: no runner involved
                continue
            assert set(ref["groups"][g][str(i)]) == set(HANDLERS)
            n += 1
    assert n >= 150


@pytest.mark.parametrize("handler", HANDLERS)
def test_oracle_results_equal_the_reference_runners(goldens, handler):
    hot, ref = goldens
    checked = 0
    for g, cases in hot["groups"].items():
        payloads = [base64.b64decode(c["payload"]) for c in cases]
        ids = [bytes.fromhex(c["task_id"]) for c in cases]
        live = loop.run_task_loop(payloads, ids, handler, keep_wire=True)          # the oracle, now
        for i, c in enumerate(cases):
            if c["wire"] is None:
                assert live[i].status == loop.REJECTED                             # Ok:false at put
                continue
            r_status, r_result, r_task_id = ref["groups"][g][str(i)][handler]
            assert live[i].wire == base64.b64decode(c["wire"])                      # same bytes the reference runner was fed
            assert live[i].status == r_status, (g, i, payloads[i][:80], r_status)
            want = None if r_result is None else base64.b64decode(r_result)
            assert live[i].result == want, (g, i, payloads[i][:80])
            # the task id on the wire is what the runner reports back
            assert json.loads(live[i].wire)["task_id"] == r_task_id
            checked += 1
    assert checked >= 150


def test_put_payload_equals_the_reference_sdks(goldens):
    hot, ref = goldens
    n = 0
    for g, per in ref["put"].items():
        for i, b64 in per.items():
            d = json.loads(base64.b64decode(hot["groups"][g][int(i)]["payload"]))
            assert loop.sdk_put_payload(*d["args"], **d["kwargs"]) == base64.b64decode(b64)
            n += 1
    assert n >= 100


def test_map_input_formatting_equals_the_reference_sdks(goldens):
    """beta9_b200.taskqueue's map() spreads inputs like the reference's Function._format_args."""
    from beta9_b200.taskqueue import _CallableWrapper
    _, ref = goldens
    assert len(ref["format_args"]) >= 10
    for case in ref["format_args"]:
        x = tuple(case["in"]["v"]) if case["in"]["t"] == "tuple" else case["in"]["v"]
        assert _CallableWrapper._format_args(x) == case["out"], case


def test_live_fuzz_against_the_reference_runner():
    """1200 random SDK-style payloads x 4 handlers through the oracle, every completion compared with what the
    reference's runner loop completed the same wire records with (tests/golden/ref_runner_fuzz_golden.json.gz,
    written by make_ref_runner_golden.py --freeze-fuzz 1200 20260921)."""
    import gzip
    from tests.golden.make_ref_runner_golden import fuzz_digest, fuzz_payloads
    with gzip.open(os.path.join(HERE, "golden", "ref_runner_fuzz_golden.json.gz")) as f:
        ref = json.load(f)
    payloads, ids = fuzz_payloads(ref["n_payloads"], ref["seed"])
    assert fuzz_digest(payloads, ids) == ref["payloads_sha256"]           # the payloads the reference runner saw
    assert sorted(ref["handlers"]) == sorted(HANDLERS)
    bad = []
    for h in HANDLERS:
        live = loop.run_task_loop(payloads, ids, h, keep_wire=True)
        assert len(live) == len(ref["handlers"][h])
        for i, (w, r) in enumerate(zip(live, ref["handlers"][h])):
            if r is None:                                                   # refused at put: no runner involved
                assert w.wire is None, (h, i)
                continue
            want = None if r[1] is None else base64.b64decode(r[1])
            if w.wire is None or w.status != r[0] or w.result != want:
                bad.append((h, i, payloads[i][:80], (w.status, w.result), (r[0], want)))
    assert not bad, bad[:5]
