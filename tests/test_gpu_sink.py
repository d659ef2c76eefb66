"""GPU: a drain whose records land as one result-sink object (b9_drain_fetch_object) holds, per task, exactly what the
reference's per-task path would have uploaded (oracle/pyoracle/resultsink.py restating pkg/task/dispatch.go:120-144 and
pkg/api/v1/task.go:295-325), and equals the object b9_sink_pack builds from records fetched the ordinary way."""
import ctypes as C

import numpy as np
import pytest

from beta9_b200 import _lib as L
from beta9_b200 import synth
from oracle import coracle
from oracle.pyoracle import loop, resultsink
from oracle.pyoracle.wire import format_uuid

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("handler", ["identity", "crc32", "json_sum"])
def test_fetch_object_matches_per_task_store(handler):
    from beta9_b200.device_queue import DeviceQueue
    lib = L.load()
    b = synth.concat([synth.strings_batch(5000, 64, adversarial_frac=0.2), synth.json_batch(200),
                      synth.from_payloads([b"", b"{}", b'{"args": [""], "kwargs": {}}', b'{"args": [0]}', b"not json"])])
    b.task_ids = synth.task_ids(b.n, seed=21)
    o = coracle.run_batch(b.task_ids, b.payload, b.offsets, handler)
    with DeviceQueue(ring_bytes=1 << 26, ring_tasks=1 << 16, max_drain_tasks=1 << 16, max_result_bytes=1 << 26) as q:
        q.push_batch(b.task_ids, b.payload, b.offsets)
        obj = q.drain_object(handler)
        assert q.depth() == 0
        # the same drain fetched the ordinary way and packed on the host gives the same records
        q.push_batch(b.task_ids, b.payload, b.offsets)
        r = q.drain(handler)
    # what the C oracle declines, the Python oracle's task loop (exact everywhere) answers
    py = np.flatnonzero(o.status == 4)
    want_st, want_res = o.status.astype(int), [o.result(i) for i in range(b.n)]
    if py.size:
        code = {"COMPLETE": 0, "ERROR": 1, "RETRY": 2, "REJECTED": 3}
        for i, w in zip(py, loop.run_task_loop([b.task(int(i)) for i in py], [b.task_ids[int(i)].tobytes() for i in py], handler)):
            want_st[i], want_res[i] = code[w.status], w.result
    store = {}
    for i in range(b.n):
        resultsink.store_task_result(store, b.task_ids[i].tobytes(), want_res[i])
    rec = L.SinkRecord()
    out = C.create_string_buffer(1 << 16)
    by_python = 0
    for i in range(b.n):
        assert lib.b9_sink_get(obj.ctypes.data, obj.size, i, C.byref(rec)) == 0
        assert C.string_at(rec.task_id, 16) == b.task_ids[i].tobytes()
        if rec.status == 4:                                  # UNSUPPORTED on the device: the host routes it through the CPU loop
            assert not rec.has_result
            continue
        by_python += int(o.status[i] == 4)
        assert rec.status == want_st[i]
        key = resultsink.task_result_path(format_uuid(b.task_ids[i].tobytes()))
        if rec.has_result:
            data = C.string_at(rec.data, rec.length)
            assert store[key] == data and data == r.result(i)
            n = lib.b9_sink_result_json(data, len(data), out, len(out))
            assert out.raw[:n] == resultsink.add_result_to_task(data)      # every device result is valid JSON: kept as it is
            assert out.raw[:n] == data
        else:
            assert key not in store
    print(f"{handler}: {by_python} device record(s) the C oracle declines checked against the Python oracle")
