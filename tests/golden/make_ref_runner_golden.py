"""Runs the REFERENCE's own runner loop over the golden wire records and freezes what it produced.

    python tests/golden/make_ref_runner_golden.py        (needs /root/reference; run from the repo root)

What is executed is the unmodified reference code, imported from /root/reference/sdk/src:
`beta9.runner.taskqueue.TaskQueueWorker.process_tasks` (sdk/src/beta9/runner/taskqueue.py:297-404) with
its `_get_next_task` (:185-204: `json.loads(task_msg)` -> Task(args, kwargs)), `FunctionHandler.__call__`
(runner/common.py:297-305) and `serialize_result` (runner/common.py:484-489). Only the gRPC stubs are
replaced (a pop that serves the golden `task_msg` bytes, a complete that records the request): that is
the process boundary. The producer side is pinned the same way: `_CallableWrapper.put`
(sdk/src/beta9/abstractions/taskqueue.py:254-295) is called with a stub that records the
`TaskQueuePutRequest.payload` it builds. Things the image lacks and that are stood in for, none on the
data path: `betterproto` (tests/golden/ref_harness/betterproto: field helpers so that the GENERATED
message classes import), `watchdog` (file-sync observer of the CLI; a mock module) and the package
`__init__` of `beta9` (it pulls the CLI's dependencies; the modules are imported directly). The user
handlers are oracle/pyoracle/handlers.py (the configs' user functions) wrapped by the reference's
`_CallableWrapper` and loaded through the reference's HANDLER=module:func mechanism
(tests/golden/ref_harness/ref_handlers.py).

The input `task_msg` bytes come from tests/golden/hot_path_golden.json, i.e. from the oracle's
restatement of Go's TaskMessage.Encode (that half stays unpinned: no Go toolchain). Output:
tests/golden/ref_runner_golden.json, checked on every CPU run by tests/test_oracle_vs_ref_runner.py.
"""
import base64
import contextlib
import importlib.abc
import importlib.machinery
import io
import json
import os
import sys
import types
from unittest import mock

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF_SDK = "/root/reference/sdk/src"
HANDLERS = ["identity", "crc32", "vadd_f32", "json_sum"]


class _MockLoader(importlib.abc.Loader):
    def create_module(self, spec):
        m = mock.MagicMock(name=spec.name)
        m.__path__, m.__name__, m.__spec__ = [], spec.name, spec
        return m

    def exec_module(self, module):
        pass


class _MockFinder(importlib.abc.MetaPathFinder):
    def find_spec(self, name, path, target=None):
        if name.split(".")[0] == "watchdog":
            return importlib.machinery.ModuleSpec(name, _MockLoader(), is_package=True)
        return None


def load_reference_runner():
    if not os.path.isdir(REF_SDK):
        raise SystemExit(f"{REF_SDK} not found: this script only runs where the reference is mounted")
    sys.meta_path.append(_MockFinder())
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden", "ref_harness"))      # the betterproto stand-in
    sys.path.insert(0, ROOT)                                                       # oracle.pyoracle.handlers
    pkg = types.ModuleType("beta9")
    pkg.__path__ = [os.path.join(REF_SDK, "beta9")]                               # skip beta9/__init__.py (CLI imports)
    sys.modules["beta9"] = pkg
    os.environ.setdefault("HANDLER", "ref_handlers:identity")
    os.environ.setdefault("STUB_ID", "7f1c2d3e-4a5b-4c6d-8e9f-0a1b2c3d4e5f")
    os.environ.setdefault("CONTAINER_ID", "taskqueue-golden-0")        # a runner container's environment (common.py:60-78)
    os.environ.setdefault("CONTAINER_HOSTNAME", "localhost")
    os.environ.setdefault("STUB_TYPE", "taskqueue")
    os.environ.setdefault("BIND_PORT", "8001")
    import beta9.runner.taskqueue as rt
    import beta9.runner.common as rc
    return rt, rc


def run_reference_worker(rt, rc, handler_name, task_msgs):
    """-> list of (task_id, task_status string, result bytes | None), one per task_msg, from the reference loop."""
    done = []

    class FakeTaskQueueStub:
        def __init__(self, channel=None):
            self.queue = list(task_msgs)

        def task_queue_pop(self, req):
            if not self.queue:
                worker.should_exit = True                       # same effect as SIGTERM (_signal_handler)
                return rt.TaskQueuePopResponse(ok=False)
            return rt.TaskQueuePopResponse(ok=True, task_msg=self.queue.pop(0))

        def task_queue_monitor(self, req):
            yield rt.TaskQueueMonitorResponse(ok=True, complete=True)

        def task_queue_complete(self, req):
            status = req.task_status
            done.append((req.task_id, getattr(status, "value", status), req.result))
            return rt.TaskQueueCompleteResponse(ok=True)

    class FakeGatewayStub:
        def __init__(self, channel=None):
            pass

    rc.config.handler = f"ref_handlers:{handler_name}"
    rt.TaskQueueServiceStub = FakeTaskQueueStub
    rt.GatewayServiceStub = FakeGatewayStub
    rt.TASK_POLLING_INTERVAL = 0
    rt.send_callback = lambda **kw: None                         # callbacks are outside this path
    import multiprocessing
    worker = rt.TaskQueueWorker(worker_index=0, parent_pid=os.getpid(), worker_startup_event=multiprocessing.Event(),
                                workers_ready=multiprocessing.Value("i", 0))
    # the reference logs every task as JSON on the process's stdout (StdoutJsonInterceptor): send fd 1 to /dev/null meanwhile
    sys.stdout.flush()
    saved, devnull = os.dup(1), os.open(os.devnull, os.O_WRONLY)
    os.dup2(devnull, 1)
    try:
        with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
            rt.TaskQueueWorker.process_tasks.__wrapped__(worker, channel=None)    # the reference loop, minus the channel factory
    finally:
        os.dup2(saved, 1)
        os.close(saved)
        os.close(devnull)
    return done


def reference_put_payload(args, kwargs):
    """The bytes the reference's `put` hands to TaskQueuePut for these Python arguments."""
    import beta9.abstractions.taskqueue as at
    import ref_handlers
    captured = []

    class Stub:
        def task_queue_put(self, req):
            captured.append(req.payload)
            return at.TaskQueuePutResponse(ok=True, task_id="00000000-0000-4000-8000-000000000000")

    w = ref_handlers.identity
    w.parent.prepare_runtime = lambda **kw: True
    w.parent.taskqueue_stub = Stub()
    w.parent.stub_id = os.environ["STUB_ID"]
    w.parent.get_client = lambda: types.SimpleNamespace(get_task_by_id=lambda i: i)
    w.put(*args, **kwargs)
    return captured[0]


def main():
    rt, rc = load_reference_runner()
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "hot_path_golden.json")))
    out = {"source": "reference runner loop (sdk/src/beta9/runner/taskqueue.py:297-404) over hot_path_golden.json wires",
           "groups": {}}
    n = 0
    for h in HANDLERS:
        msgs, where = [], []
        for gname, cases in golden["groups"].items():
            for i, c in enumerate(cases):
                if c["wire"] is None:                           # refused at put (Ok:false): never reaches a runner
                    continue
                msgs.append(base64.b64decode(c["wire"]))
                where.append((gname, i))
        done = run_reference_worker(rt, rc, h, msgs)
        assert len(done) == len(msgs), (h, len(done), len(msgs))
        for (gname, i), (task_id, status, result) in zip(where, done):
            slot = out["groups"].setdefault(gname, {}).setdefault(str(i), {})
            slot[h] = [str(status), None if result is None else base64.b64encode(result).decode(), task_id]
            n += 1
    # producer side: every golden payload that is a plain {"args": [...], "kwargs": {...}} document, through put()
    out["put"] = {}
    for gname, cases in golden["groups"].items():
        for i, c in enumerate(cases):
            try:
                d = json.loads(base64.b64decode(c["payload"]))
            except Exception:
                continue
            if not (isinstance(d, dict) and set(d) == {"args", "kwargs"} and isinstance(d["args"], list) and isinstance(d["kwargs"], dict)):
                continue
            out["put"].setdefault(gname, {})[str(i)] = base64.b64encode(reference_put_payload(d["args"], d["kwargs"])).decode()
            n += 1
    # Function.map's input formatting (sdk/src/beta9/abstractions/function.py:246-251), for the SDK mirror's map()
    import beta9.abstractions.function as fn
    samples = [{"t": "value", "v": 5}, {"t": "value", "v": "s"}, {"t": "tuple", "v": [1, 2]}, {"t": "list", "v": [3, 4]},
               {"t": "tuple", "v": [[1], {"k": 2}]}, {"t": "value", "v": {"d": 1}}, {"t": "value", "v": None},
               {"t": "tuple", "v": []}, {"t": "list", "v": []}, {"t": "tuple", "v": [[1, 2]]}, {"t": "list", "v": [[1, 2], 3]}]
    out["format_args"] = []
    for smp in samples:
        x = tuple(smp["v"]) if smp["t"] == "tuple" else smp["v"]
        out["format_args"].append({"in": smp, "out": fn._CallableWrapper._format_args(None, x)})
    path = os.path.join(ROOT, "tests", "golden", "ref_runner_golden.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print(path, n, "task executions through the reference runner")


def fuzz_payloads(n_payloads: int, seed: int):
    """-> (payloads, task ids): random SDK-style put payloads, the same ones for the same (n_payloads, seed)."""
    import random
    sys.path.insert(0, ROOT)
    from oracle.pyoracle import loop
    rnd = random.Random(seed)
    alphabet = ["a", "Z", "0", " ", '"', "\\", "/", "<", ">", "&", "\n", "\t", "\x01", "\x7f", "\u00e9", "\u2028", "\u20ac",
                "\U0001f600", "\ud83d", "\udc00", "values", "=", "+"]

    def rstr():
        return "".join(rnd.choice(alphabet) for _ in range(rnd.randint(0, 12)))

    def rval(depth=0):
        k = rnd.randint(0, 9 if depth < 2 else 5)
        if k == 0: return None
        if k == 1: return rnd.choice([True, False])
        if k == 2: return rnd.randint(-10**rnd.randint(0, 17), 10**rnd.randint(0, 17))
        if k == 3: return rnd.choice([0.0, 0.5, -1.25, 1e21, 1e-7, 3.14159, 2.0**60, 123456789.125])
        if k in (4, 5): return rstr()
        if k in (6, 7): return [rval(depth + 1) for _ in range(rnd.randint(0, 4))]
        return {rstr(): rval(depth + 1) for _ in range(rnd.randint(0, 3))}

    payloads = []
    for i in range(n_payloads):
        shape = rnd.randint(0, 5)
        if shape == 0: args, kwargs = (rstr(),), {}
        elif shape == 1: args, kwargs = ({"values": [rnd.randint(0, 10**6) for _ in range(rnd.randint(0, 6))], "id": i},), {}
        elif shape == 2:
            raw = bytes(rnd.randrange(256) for _ in range(8 * rnd.randint(0, 4)))
            args, kwargs = (base64.b64encode(raw).decode(),), {}
        elif shape == 3: args, kwargs = tuple(rval() for _ in range(rnd.randint(0, 3))), {}
        else: args, kwargs = tuple(rval() for _ in range(rnd.randint(0, 2))), {rstr(): rval() for _ in range(rnd.randint(0, 2))}
        payloads.append(loop.sdk_put_payload(*args, **kwargs))
    return payloads, [rnd.randbytes(16) for _ in payloads]


def fuzz(n_payloads: int, seed: int) -> int:
    """Live check (no files written): random SDK-style payloads -> the oracle's wire records -> the
    reference runner; every status / result must equal the oracle's. Returns the number of mismatches."""
    rt, rc = load_reference_runner()
    from oracle.pyoracle import loop
    payloads, ids = fuzz_payloads(n_payloads, seed)
    bad = 0
    for h in HANDLERS:
        want = loop.run_task_loop(payloads, ids, h, keep_wire=True)
        live = [w for w in want if w.wire is not None]
        done = run_reference_worker(rt, rc, h, [w.wire for w in live])
        assert len(done) == len(live)
        for w, (task_id, status, result) in zip(live, done):
            if w.status != str(status) or w.result != result:
                bad += 1
                sys.stderr.write(f"MISMATCH handler={h} wire={w.wire[:200]!r} oracle=({w.status},{w.result!r}) reference=({status},{result!r})\n")
    print(f"fuzz: {n_payloads} payloads x {len(HANDLERS)} handlers through the reference runner, {bad} mismatches")
    return bad


def fuzz_digest(payloads, ids) -> str:
    import hashlib
    h = hashlib.sha256()
    for p, i in zip(payloads, ids):
        h.update(i); h.update(len(p).to_bytes(8, "little")); h.update(p)
    return h.hexdigest()


def freeze_fuzz(n_payloads: int, seed: int) -> None:
    """What the reference runner completed the wire records of fuzz_payloads(n_payloads, seed) with ->
    tests/golden/ref_runner_fuzz_golden.json.gz, which tests/test_oracle_vs_ref_runner.py compares the oracle with.
    The payloads themselves are regenerated from the seed; their digest is stored to catch a changed generator."""
    import gzip
    rt, rc = load_reference_runner()
    from oracle.pyoracle import loop
    payloads, ids = fuzz_payloads(n_payloads, seed)
    out = {"source": "reference runner loop (sdk/src/beta9/runner/taskqueue.py:297-404) over the oracle's wire records",
           "n_payloads": n_payloads, "seed": seed, "payloads_sha256": fuzz_digest(payloads, ids), "handlers": {}}
    for h in HANDLERS:
        live = loop.run_task_loop(payloads, ids, h, keep_wire=True)
        done = iter(run_reference_worker(rt, rc, h, [w.wire for w in live if w.wire is not None]))
        # one entry per payload: None where put refused it (no task, no runner), else what the runner completed it with
        per = []
        for w in live:
            if w.wire is None:
                per.append(None)
                continue
            _, status, result = next(done)
            per.append([str(status), None if result is None else base64.b64encode(result).decode()])
        assert next(done, None) is None
        out["handlers"][h] = per
    path = os.path.join(ROOT, "tests", "golden", "ref_runner_fuzz_golden.json.gz")
    with gzip.GzipFile(path, "wb", mtime=0) as f:
        f.write(json.dumps(out, sort_keys=True).encode())
    print(path, n_payloads, "payloads x", len(HANDLERS), "handlers through the reference runner")


if __name__ == "__main__":
    if len(sys.argv) >= 3 and sys.argv[1] == "--fuzz":
        sys.exit(1 if fuzz(int(sys.argv[2]), int(sys.argv[3]) if len(sys.argv) > 3 else 0xB9) else 0)
    if len(sys.argv) >= 3 and sys.argv[1] == "--freeze-fuzz":
        freeze_fuzz(int(sys.argv[2]), int(sys.argv[3]) if len(sys.argv) > 3 else 0xB9)
        sys.exit(0)
    main()
