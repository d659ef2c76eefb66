"""Every handler on each way a warp-tile's bytes reach the drain kernel, against the oracle.

drain3_kernel (beta9_b200/csrc/drain2.cuh) gets a tile of `tt` tasks to its handler code in one of four ways:
  whole      the tasks are contiguous in the ring and their 16-byte hull fits the stage buffer (`in_cap`): one bulk copy;
  scattered  they are not contiguous (the tile spans two pushes, or the ring's end) but the sum of their per-task
             16-byte hulls fits: one bulk copy per task;
  per-task   crc32 / json_sum only, when neither fits: one task at a time, if `mis + len + 16 <= in_cap`;
  global     otherwise: generic loads from the ring.
`in_cap` comes from launch_drain3 (b9gpu.cu) or from B9_STAGE_BYTES, read at context creation. `tile_paths` restates the
choice and `RingModel` restates where pushes land (ring_place.h), so that every scenario can show which paths it reached;
the census is printed under -s and its floors are checked by the last test of the file.
"""
import json
from collections import Counter, deque
from dataclasses import dataclass

import numpy as np
import pytest

from beta9_b200 import synth
from oracle import coracle
from tests.test_ring_place import script  # noqa: F401  (fixture: ring_place.h built for the host)

HANDLERS = ["identity", "crc32", "vadd_f32", "json_sum"]
TF_CANCELLED, TF_HTTP, TF_PICKLE = 0x01, 0x02, 0x04
SEG_ALIGN = 256                                   # ring_place.h B9_SEG_ALIGN
TILE = {"identity": 32, "crc32": 4, "vadd_f32": 32, "json_sum": 4}     # json_sum: 4 for windows below json_tile_bound()
PATHS = ("whole", "scattered", "per-task", "global")
KERNEL_PATHS = {h: PATHS if h in ("crc32", "json_sum") else ("whole", "scattered", "global") for h in HANDLERS}
STAGE_SIZES = [1024, 2048, 5120, 16384, 49152, None]     # None: the size launch_drain3 derives from the window
CENSUS_FLOOR = 300
MAX_TASK_BYTES = 1 << 20                          # b9_ctx_create's default max_task_bytes

CENSUS = Counter()                                # (handler, path) -> ready tasks drained that way, over the whole file
BOUNDARY = []                                     # (handler, case, path the arithmetic predicts, path the census gave)
RAN = set()


# ---------------------------------------------------------------- where pushes land (ring_place.h, b9gpu.cu push_impl)
def seg_span(nbytes):
    return (nbytes + SEG_ALIGN - 1) & ~(SEG_ALIGN - 1)


def ring_place(ring_bytes, have_segments, oldest, wp, live_bytes, nbytes):
    """b9_ring_place: the start of a new segment of `nbytes`, or None when the ring cannot take it now."""
    need = seg_span(nbytes)
    if need > ring_bytes:
        return None
    if not have_segments:
        return 0
    if live_bytes == 0:
        return wp if wp + need <= ring_bytes else 0
    if wp == oldest:
        return wp if need == 0 else None
    if wp > oldest:
        if wp + need <= ring_bytes:
            return wp
        return 0 if need <= oldest else None
    return wp if wp + need <= oldest else None


class RingModel:
    """The library's push / drain bookkeeping: segments in FIFO order, each freed once the head has passed all of its
    tasks, the write position back at 0 when none is left; a push is refused when the slot ring or the payload ring
    cannot take it."""

    def __init__(self, ring_bytes, ring_tasks):
        self.ring_bytes, self.ring_tasks = ring_bytes, ring_tasks
        self.segs = deque()                       # [first_task, n, start, nbytes, max_len]
        self.wp = self.head = self.tail = 0
        self.wraps = 0                            # pushes placed below the write position: the payload ring wrapped

    def _free(self):
        while self.segs and self.segs[0][0] + self.segs[0][1] <= self.head:
            self.segs.popleft()
        if not self.segs:
            self.wp = 0

    def push(self, lens):
        """-> the new segment's physical start, or None where b9_batch_push answers B9_ENOSPC."""
        self._free()
        n, nbytes = len(lens), int(sum(lens))
        if n > self.ring_tasks - (self.tail - self.head):
            return None
        live = sum(s[3] for s in self.segs)
        start = ring_place(self.ring_bytes, bool(self.segs), self.segs[0][2] if self.segs else 0, self.wp, live, nbytes)
        if start is None:
            return None
        self.wraps += start < self.wp
        self.segs.append([self.tail, n, start, nbytes, min(max(lens, default=0), MAX_TASK_BYTES)])
        self.wp = start + seg_span(nbytes)
        self.tail += n
        return start

    def pop(self, k):
        self.head += min(k, self.tail - self.head)
        self._free()

    def window_max_len(self, n):
        """The longest task of the segments a window of n tasks touches; 0 (unknown) if one of them says 0."""
        lo, hi = self.head, self.head + n
        ms = [s[4] for s in self.segs if max(lo, s[0]) < min(hi, s[0] + s[1])]
        return 0 if (not ms or 0 in ms) else max(ms)


# ---------------------------------------------------------------- which path each tile takes (drain3_kernel, launch_drain3)
def derived_in_cap(handler, in_bytes, n, max_len, override):
    """launch_drain3's stage size for a window: B9_STAGE_BYTES rounded up to 1 KiB, or the average task x tt x 1.1 + 768
    (x 1.35 for crc32) within [1 KiB, 48 KiB], capped at max_len x tt + 32 except for crc32, rounded up to 128."""
    if override:
        return (override + 1023) & ~1023
    tt, avg = TILE[handler], in_bytes // n
    want = avg * tt * 27 // 20 + 768 if handler == "crc32" else avg * tt * 11 // 10 + 768
    cap = min(48 << 10, max(1 << 10, want))
    if handler != "crc32" and max_len:
        cap = min(cap, max(1 << 10, max_len * tt + 32))
    return (cap + 127) & ~127


def tile_metrics(offs, lens):
    """-> (contiguous, 16-byte hull of the whole tile, sum of the per-task 16-byte hulls)."""
    o, e = offs.astype(np.int64), (offs + lens).astype(np.int64)
    contig = bool(np.all(o[1:] == e[:-1]))
    hull = int(((e[-1] + 15) & ~15) - (o[0] & ~15))
    scat = int(np.where(lens > 0, ((e + 15) & ~15) - (o & ~15), 0).sum())
    return contig, hull, scat


def tile_paths(handler, offs, lens, flags, in_cap):
    """The path of every task of a window: "whole" / "scattered" for a staged tile; otherwise "per-task" or "global"
    by task (crc32 and json_sum), or "global"; "cancelled" for cancelled slots, "none" for tasks whose bytes are not
    read (pickle-framed tasks under crc32 / json_sum / vadd_f32)."""
    tt, n = TILE[handler], len(lens)
    out = []
    for t0 in range(0, n, tt):
        o, ln, fl = offs[t0:t0 + tt], lens[t0:t0 + tt], flags[t0:t0 + tt]
        contig, hull, scat = tile_metrics(o, ln)
        staged = ("whole" if hull <= in_cap else None) if contig else ("scattered" if scat <= in_cap else None)
        for k in range(len(ln)):
            f = int(fl[k])
            if f & TF_CANCELLED:
                out.append("cancelled")
            elif handler != "identity" and f & TF_PICKLE:
                out.append("none")
            elif staged:
                out.append(staged)
            elif handler in ("crc32", "json_sum") and not f & TF_HTTP:
                out.append("per-task" if (int(o[k]) & 15) + int(ln[k]) + 16 <= in_cap else "global")
            else:
                out.append("global")
    return out


def json_tile_bound():
    """launch_drain3 gives json_sum tiles of 4 documents while ceil(n / 8) < 3 x CTAs per SM x SMs x 2 warps; one CTA
    per SM always fits, so windows with fewer 8-document tiles than 6 x SMs are safe."""
    import torch
    return 6 * torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------- tasks
@dataclass
class Task:
    payload: bytes
    kind: str                       # "str" "vadd" "json" "http" "pickle"
    flag: int = 0
    tid: bytes = b""
    off: int = 0                    # physical start in the payload ring
    ts: int = 0
    exp: int = 0
    retries: int = 0


def tasks_of(batch, kind, flag=0):
    return [Task(batch.task(i), kind, flag) for i in range(batch.n)]


FRAME = len(synth.PREFIX) + len(synth.SUFFIX)     # 28 bytes around a string argument


def string_task(length, ch=b"x"):
    """An SDK-framed string argument of exactly `length` bytes (>= FRAME)."""
    assert length >= FRAME
    return Task(synth.PREFIX + ch * (length - FRAME) + synth.SUFFIX, "str")


def json_task(length, seed=0):
    """A json_sum document task of exactly `length` bytes (>= 80)."""
    vals = [(seed * 7919 + 13 * j) % 1000003 for j in range(4)]
    p = json.dumps({"args": [{"v": vals, "p": ""}], "kwargs": {}}).encode()
    return Task(p.replace(b'"p": ""', b'"p": "' + b"y" * (length - len(p)) + b'"'), "json")


def http_tasks():
    from tests.test_gpu_parity import _http_bodies
    return [Task(b, "http", TF_HTTP) for b in _http_bodies()]


def pickle_tasks(rng, n):
    from oracle.pyoracle import funcloop
    pool = ["a", "Z", " ", '"', "\\", "\n", "é", "€", "\U0001f600"]
    out = []
    for k in range(n):
        m = int(rng.choice([0, 1, 5, 15, 16, 17, 40, 100, 255, 256, 700, 3000]))
        s = "".join(chr(int(c)) for c in rng.integers(0x20, 0x7F, m)) if k % 4 else "".join(pool[int(j)] for j in rng.integers(0, len(pool), m))
        out.append(Task(funcloop.frame_map_input(s), "pickle", TF_PICKLE))
    return out


def own_shape(handler, rng, n):
    """The handler's own configuration shape (BASELINE configs), at varied sizes."""
    if handler == "identity":
        return tasks_of(synth.strings_batch(n, int(rng.choice([1, 64, 256])), adversarial_frac=0.05, seed=int(rng.integers(1 << 30))), "str")
    if handler == "crc32":
        return tasks_of(synth.crc_batch(n, seed=int(rng.integers(1 << 30))), "str")
    if handler == "vadd_f32":
        return tasks_of(synth.vadd_batch(n, floats_per_vec=int(rng.choice(list(range(1, 14)) + [64])), seed=int(rng.integers(1 << 30))), "vadd")
    return tasks_of(synth.json_batch(n, doc_bytes=int(rng.choice([200, 500, 1024, 2000, 4096])), seed=int(rng.integers(1 << 30))), "json")


def mixed_pool(handler, rng):
    """Payloads of every configuration's shape, the handler's own weighted up."""
    pool = own_shape(handler, rng, 300) + own_shape(handler, rng, 300)
    pool += tasks_of(synth.strings_batch(150, int(rng.integers(1, 120)), adversarial_frac=0.3, seed=int(rng.integers(1 << 30))), "str")
    pool += tasks_of(synth.crc_batch(100, seed=int(rng.integers(1 << 30))), "str")
    pool += tasks_of(synth.vadd_batch(100, floats_per_vec=int(rng.integers(1, 14)), seed=int(rng.integers(1 << 30))), "vadd")
    pool += tasks_of(synth.vadd_special_batch(50, floats_per_vec=int(rng.integers(1, 14)), seed=int(rng.integers(1 << 30))), "vadd")
    pool += tasks_of(synth.json_batch(60, doc_bytes=int(rng.choice([150, 300, 700])), seed=int(rng.integers(1 << 30))), "json")
    pool += [Task(b"", "str"), Task(b"{}", "str")] * 10
    return pool


def copy_task(t, flag=None):
    return Task(t.payload, t.kind, t.flag if flag is None else flag)


# ---------------------------------------------------------------- a queue and what the test knows about it
class Queue:
    """A DeviceQueue, its pending tasks in FIFO order with their physical offsets, and the ring model. Every drain
    restates each tile's path (counted into CENSUS) and checks every record against the oracle."""
    _next_id = 0

    def __init__(self, ring_bytes=1 << 26, ring_tasks=1 << 15, stage_bytes=None, max_result_bytes=1 << 27):
        from beta9_b200.device_queue import DeviceQueue
        self.q = DeviceQueue(ring_bytes=ring_bytes, ring_tasks=ring_tasks, max_drain_tasks=ring_tasks, max_result_bytes=max_result_bytes)
        self.model = RingModel(ring_bytes, ring_tasks)
        self.stage_bytes = stage_bytes
        self.pending = deque()

    def close(self):
        self.q.close()

    def push(self, tasks, meta=False):
        from beta9_b200 import _lib as L
        n = len(tasks)
        ids = synth.task_ids(n, seed=0x57A6E, start=Queue._next_id)
        Queue._next_id += n
        b = synth.from_payloads([t.payload for t in tasks])
        kw = dict(flags=np.array([t.flag for t in tasks], np.uint8))
        if meta:
            kw.update(timestamp_unix=np.array([t.ts for t in tasks], np.int64), expires_unix_ns=np.array([t.exp for t in tasks], np.int64),
                      retries=np.array([t.retries for t in tasks], np.uint8))
        start = self.model.push([len(t.payload) for t in tasks])
        try:
            self.q.push_batch(ids, b.payload, b.offsets, **kw)
        except L.B9Error as e:
            assert e.code == L.B9_ENOSPC and start is None, (e, start)
            return False
        assert start is not None, "the library took a push the ring model refuses"
        for i, t in enumerate(tasks):
            t.tid, t.off = ids[i].tobytes(), start + int(b.offsets[i])
        self.pending.extend(tasks)
        assert self.q.depth() == len(self.pending)
        return True

    def window(self, max_tasks):
        return [self.pending[i] for i in range(min(max_tasks, len(self.pending)))]

    def paths(self, handler, win):
        lens = np.array([len(t.payload) for t in win], np.int64)
        in_cap = derived_in_cap(handler, int(lens.sum()), len(win), self.model.window_max_len(len(win)), self.stage_bytes)
        offs = np.array([t.off for t in win], np.int64)
        return tile_paths(handler, offs, lens, np.array([t.flag for t in win], np.uint8), in_cap)

    def drain(self, handler, max_tasks=1 << 22, peek=False):
        """Drains (or peeks) up to max_tasks through `handler`, checks every record; -> (DrainResult, paths of the window)."""
        win = self.window(max_tasks)
        if handler == "json_sum":
            assert (len(win) + 7) // 8 < json_tile_bound(), "json_sum window too large for tiles of 4"
        paths = self.paths(handler, win)
        if peek:
            assert self.q.drain_launch(handler, max_tasks, peek=True) == sum(1 for t in win if not t.flag & TF_CANCELLED)
            r = self.q.fetch()
        else:
            r = self.q.drain(handler, max_tasks=max_tasks)
        assert r.n_popped == len(win)
        check_records(handler, win, r)
        if not peek:
            for _ in win:
                self.pending.popleft()
            self.model.pop(len(win))
            assert self.q.depth() == len(self.pending)
            CENSUS.update((handler, p) for p in paths if p in PATHS)
        return r, paths

    def drain_all(self, handler, **kw):
        return self.drain(handler, max_tasks=len(self.pending), **kw)


def sub_result(r, idx):
    from beta9_b200.device_queue import DrainResult
    return DrainResult(r.task_ids[idx], r.status[idx], r.has_result[idx], r.offsets[idx], r.lengths[idx], r.payload, len(idx))


def check_records(handler, win, r):
    """Every record of a drain: FIFO order without the cancelled slots; SDK payloads against the C oracle (the Python one
    where it declines) through test_gpu_parity's assert_matches_oracle, HTTP bodies and pickle-framed tasks against the
    Python oracles."""
    from oracle.pyoracle import funcloop, loop
    from tests.test_gpu_parity import assert_matches_oracle
    keep = [t for t in win if not t.flag & TF_CANCELLED]
    assert r.n == len(keep)
    assert [r.task_ids[i].tobytes() for i in range(r.n)] == [t.tid for t in keep], "records out of FIFO order"
    plain = np.array([i for i, t in enumerate(keep) if t.kind not in ("http", "pickle")], np.int64)
    if plain.size:
        sb = synth.from_payloads([keep[i].payload for i in plain])
        sb.task_ids = np.stack([np.frombuffer(keep[i].tid, np.uint8) for i in plain])
        o = coracle.run_batch(sb.task_ids, sb.payload, sb.offsets, handler, nthreads=8)
        json_docs = [j for j, i in enumerate(plain) if keep[i].kind == "json"]
        # identity declines a non-string argument (json_sum's documents) and never answers it wrong
        allow = len(json_docs) if handler == "identity" else 0
        sr = sub_result(r, plain)
        decided = np.flatnonzero((sr.status != 4) & (o.status != 4))
        wrong = [int(i) for i in decided if (int(sr.status[i]), sr.result(int(i))) != (int(o.status[i]), o.result(int(i)))]
        assert not wrong, f"{handler}: {len(wrong)} of {len(plain)} records wrong, first at {wrong[:5]}"
        assert_matches_oracle(sb, sr, o, allow_unsupported=allow)
        assert set(np.flatnonzero(sr.status == 4).tolist()) <= set(json_docs)
    code = {"COMPLETE": 0, "ERROR": 1, "RETRY": 2, "REJECTED": 3}
    http = [i for i, t in enumerate(keep) if t.kind == "http"]
    if http:
        want = loop.run_task_loop([keep[i].payload for i in http], [keep[i].tid for i in http], handler, http_body=True)
        declined = 0
        for i, w in zip(http, want):
            if r.status[i] == 4:                   # floats etc.: the device declines, never guesses
                assert not r.has_result[i]
                declined += 1
                continue
            assert (int(r.status[i]), r.result(i)) == (code[w.status], w.result), keep[i].payload
        assert declined <= len(http) // 10 + 1
    for i, t in enumerate(keep):
        if t.kind != "pickle":
            continue
        if handler == "identity":
            st, want = funcloop.run_function_task(t.payload, "identity")
            assert st == funcloop.COMPLETE and (int(r.status[i]), r.result(i)) == (0, want), t.payload[:80]
        else:                                      # the function path is identity only
            assert int(r.status[i]) == 4 and r.result(i) is None


def census_line(handler, paths):
    c = Counter(p for p in paths if p in PATHS)
    return f"{handler:9s} " + " ".join(f"{p}={c[p]}" for p in PATHS)


@pytest.fixture
def stage(monkeypatch):
    """make(stage_bytes, **queue_args) -> a Queue whose context was created under B9_STAGE_BYTES = stage_bytes (unset
    for None); the variable is restored afterwards and every queue closed."""
    made = []

    def make(stage_bytes, **kw):
        if stage_bytes is None:
            monkeypatch.delenv("B9_STAGE_BYTES", raising=False)
        else:
            monkeypatch.setenv("B9_STAGE_BYTES", str(stage_bytes))
        q = Queue(stage_bytes=stage_bytes, **kw)
        made.append(q)
        return q
    yield make
    for q in made:
        q.close()


# ---------------------------------------------------------------- the placement restatement against ring_place.h (CPU)
def test_ring_model_matches_ring_place_shim(script):
    """RingModel's starts and refusals equal those of the library's own placement function (ring_place.h compiled for
    the host, as test_ring_place.py builds it) on random scripts of pushes and partial drains; the shim pops a segment
    when the model's head has passed all of its tasks."""
    for seed in range(12):
        rng = np.random.default_rng(1000 + seed)
        ring = int(rng.choice([1024, 4096, 1 << 16]))
        m = RingModel(ring, 1 << 30)
        ops, want = [], []
        for _ in range(1500):
            if rng.random() < 0.5:
                n = int(rng.integers(1, 6))
                k = rng.random()
                if k < 0.4:
                    lens = [0] * (n - 1) + [256 * int(rng.integers(1, max(2, ring // 512)))]
                elif k < 0.9:
                    lens = rng.integers(0, max(2, ring // (2 * n)), n).tolist()
                else:
                    lens = [0] * n
                s = m.push(lens)
                ops.append(sum(lens) + 1)
                want.append(-1 if s is None else s)
            else:
                before = len(m.segs)
                m.pop(int(rng.integers(0, 8)))
                for _ in range(before - len(m.segs)):
                    ops.append(0)
                    want.append(0)
        got = script(ring, ops)
        assert got == want, seed
        assert m.wraps > 0 or ring == 1 << 16


# ---------------------------------------------------------------- 1. forced stage sizes
@pytest.mark.gpu
@pytest.mark.parametrize("h", HANDLERS)
@pytest.mark.parametrize("stage_bytes", STAGE_SIZES)
def test_forced_stage_sizes(stage, stage_bytes, h):
    """Each configuration's shape, escape-dense strings, special floats, HTTP bodies, pickle-framed tasks and 7 % cancelled
    slots, one push each into an empty ring and drained whole, at forced stage sizes and at the derived one."""
    q = stage(stage_bytes)
    rng = np.random.default_rng(stage_bytes or 7)
    batches = []
    if h == "identity":
        batches += [tasks_of(synth.strings_batch(2000, 64, adversarial_frac=0.05, seed=3), "str"),
                    tasks_of(synth.strings_batch(500, 256, adversarial_frac=0.05, seed=4), "str")]
    elif h == "crc32":
        batches += [tasks_of(synth.crc_batch(1500, seed=5), "str"),
                    tasks_of(synth.crc_batch(300, seed=6, lengths=rng.integers(900, 4097, 300)), "str")]
    elif h == "vadd_f32":
        batches += [tasks_of(synth.vadd_batch(120, floats_per_vec=f, seed=f), "vadd") for f in list(range(1, 14)) + [64]]
        batches += [tasks_of(synth.vadd_special_batch(120, floats_per_vec=f, seed=f), "vadd") for f in (1, 2, 3, 7, 32)]
    else:
        batches += [tasks_of(synth.json_batch(150, doc_bytes=d, seed=d), "json") for d in (200, 700, 1024, 2048, 4096)]
    batches.append(tasks_of(synth.strings_batch(400, 100, adversarial_frac=1.0, seed=6), "str"))     # escape-dense
    batches.append(http_tasks())
    batches.append(pickle_tasks(rng, 300))
    own = own_shape(h, rng, 1200)
    gone = rng.random(len(own)) < 0.07
    batches.append([copy_task(t, TF_CANCELLED if g else 0) for t, g in zip(own, gone)])
    paths = []
    for b in batches:
        assert q.push(b)
        paths += q.drain_all(h)[1]
    print(f"\nstage {stage_bytes}: " + census_line(h, paths), end="")
    RAN.add(f"stage{stage_bytes}{h}")


# ---------------------------------------------------------------- 2. windows across pushes
def push_run(q, pool, rng, n_pushes, cancel_frac=0.05):
    """n_pushes small pushes of pool tasks; every fourth one is topped up to a multiple of 256 bytes with a string
    task, so that the next push starts right behind it and the tile across them is contiguous."""
    for k in range(n_pushes):
        m = int(rng.integers(1, 41))
        ts = [copy_task(pool[int(i)], TF_CANCELLED if rng.random() < cancel_frac else 0) for i in rng.integers(0, len(pool), m)]
        if k % 4 == 3:
            total = sum(len(t.payload) for t in ts)
            ts.append(string_task(FRAME + (-(total + FRAME)) % 256 + 256 * int(rng.integers(0, 2))))
            assert sum(len(t.payload) for t in ts) % 256 == 0
        assert q.push(ts)


@pytest.mark.gpu
@pytest.mark.parametrize("h", HANDLERS)
@pytest.mark.parametrize("stage_bytes", [None, 16384, 49152])
def test_windows_across_pushes(stage, stage_bytes, h):
    """20 to 60 pushes of 1 to 40 tasks of every shape, some cancelled, drained as one window: nearly every tile spans
    two pushes; a push topped up to a multiple of 256 bytes makes the tile behind it contiguous."""
    q = stage(stage_bytes)
    rng = np.random.default_rng(100 * HANDLERS.index(h) + (stage_bytes or 0) % 997)
    pool = mixed_pool(h, rng)
    paths = []
    for _ in range(4):
        push_run(q, pool, rng, int(rng.integers(20, 61)))
        paths += q.drain_all(h)[1]
    print(f"\nacross pushes, stage {stage_bytes}: " + census_line(h, paths), end="")
    RAN.add(f"across{stage_bytes}{h}")


# ---------------------------------------------------------------- 3. partial windows
@pytest.mark.gpu
@pytest.mark.parametrize("h", HANDLERS)
@pytest.mark.parametrize("stage_bytes", [None, 5120])
def test_partial_windows(stage, stage_bytes, h):
    """Windows that end (and so the next one starts) inside a push: tiles aligned to the head, not to the segment."""
    q = stage(stage_bytes)
    rng = np.random.default_rng(31 + len(h))
    pool = mixed_pool(h, rng)
    paths = []
    for _ in range(3):
        for _ in range(8):
            assert q.push([copy_task(pool[int(i)], TF_CANCELLED if rng.random() < 0.05 else 0)
                           for i in rng.integers(0, len(pool), int(rng.integers(50, 300)))])
        for take in (1, 7, 33, 101, 250, int(rng.integers(1, 500)), 3, 65):
            paths += q.drain(h, max_tasks=take)[1]
        paths += q.drain_all(h)[1]
        assert not q.pending
    print(f"\npartial windows, stage {stage_bytes}: " + census_line(h, paths), end="")
    RAN.add(f"partial{stage_bytes}{h}")


# ---------------------------------------------------------------- 4. ring wrap, with wire records and expiry
NOW = coracle.DEFAULT_NOW_NS
TTL = 7200


def wire_oracle(t):
    """TaskMessage.Encode of one pending task with its own timestamp, expiry and retries (0 expiry = Go's zero time);
    None where the reference would not have created the task."""
    from oracle.pyoracle.gojson import GO_ZERO_TIME_UNIX_NS, GoJSONError
    from oracle.pyoracle.loop import go_unmarshal_task_payload
    from oracle.pyoracle.wire import TaskMessage, TaskPolicy, format_uuid
    try:
        args, kwargs = go_unmarshal_task_payload(t.payload)
    except GoJSONError:
        return None
    pol = TaskPolicy(max_retries=3, timeout=3600, expires_unix_ns=t.exp or GO_ZERO_TIME_UNIX_NS, ttl=TTL)
    return TaskMessage(task_id=format_uuid(t.tid), workspace_name=coracle.DEFAULT_WS, stub_id=coracle.DEFAULT_STUB,
                       executor="taskqueue", args=args, kwargs=kwargs, policy=pol, retries=t.retries, timestamp=t.ts).encode()


def check_wire(q, k):
    r = q.q.wire_encode(coracle.DEFAULT_WS, coracle.DEFAULT_STUB, max_tasks=k, ttl=TTL)
    win = q.window(k)
    assert r.n == len(win) and q.q.depth() == len(q.pending)          # a peek
    assert [r.task_ids[i].tobytes() for i in range(r.n)] == [t.tid for t in win]
    decided = 0
    for i, t in enumerate(win):
        if r.status[i] == 4:                        # json_sum's documents (keys not in sorted order): declined, never guessed
            assert r.result(i) is None and t.kind == "json", t.payload[:80]
            continue
        want = wire_oracle(t)
        if want is None:
            assert r.status[i] == 3 and r.result(i) is None, t.payload[:80]
        else:
            assert r.status[i] == 0 and r.result(i) == want, (t.payload[:80], r.result(i), want)
            decided += 1
    return decided


@pytest.mark.gpu
def test_ring_wrap_all_handlers_with_wire_records_and_expiry(stage):
    """A 2 MiB payload ring and a 2048-slot ring, pushes of every shape with per-task timestamps, expiries (0, negative,
    sub-second, past and future) and retries, partial drains by every handler in turn, until both rings have wrapped
    several times; wire records and expire() are checked on the wrapped rings."""
    q = stage(None, ring_bytes=2 << 20, ring_tasks=2048, max_result_bytes=1 << 26)
    rng = np.random.default_rng(2024)
    pools = {h: mixed_pool(h, rng) for h in HANDLERS}
    paths = {h: [] for h in HANDLERS}
    refused = wires = expired_total = 0
    step = 0
    while (q.model.wraps < 5 or q.model.tail < 5 * 2048) and step < 400:
        h = HANDLERS[step % 4]
        pool = pools[HANDLERS[(step // 4) % 4]]
        ts = []
        for i in rng.integers(0, len(pool), int(rng.integers(1, 400))):
            t = copy_task(pool[int(i)], TF_CANCELLED if rng.random() < 0.03 else 0)
            t.ts = int(rng.choice([NOW // 10**9 + int(rng.integers(-10**6, 10**6)), int(rng.integers(-10**10, 0)), 0, int(rng.integers(0, 10**9))]))
            t.exp = int(rng.choice([0, -int(rng.integers(1, 10**18)), int(rng.integers(1, 10**9)), NOW - int(rng.integers(1, 10**15)),
                                    NOW + int(rng.integers(1, 10**15)), NOW]))
            t.retries = int(rng.integers(0, 256))
            ts.append(t)
        if not q.push(ts, meta=True):
            refused += 1
        if step % 5 == 0 and q.pending:
            wires += check_wire(q, int(rng.integers(1, min(len(q.pending), 600) + 1)))
        if step % 7 == 3:
            gone = [t for t in q.pending if not t.flag & TF_CANCELLED and t.exp != 0 and t.exp <= NOW]
            assert q.q.expire(NOW) == len(gone)
            for t in gone:
                t.flag |= TF_CANCELLED
            expired_total += len(gone)
        take = int(rng.integers(1, 300))
        paths[h] += q.drain(h, max_tasks=take)[1]
        step += 1
    while q.pending:
        paths["identity"] += q.drain("identity", max_tasks=1000)[1]
    assert q.model.wraps >= 5 and q.model.tail >= 5 * 2048, (q.model.wraps, q.model.tail)
    assert refused > 0 and wires > 1000 and expired_total > 100, (refused, wires, expired_total)
    assert q.q.depth() == 0 and q.q.depth_bytes() == 0
    print(f"\nring wrap: {step} steps, {q.model.wraps} payload-ring wraps, {q.model.tail} tasks over 2048 slots, {refused} pushes refused, "
          f"{wires} wire records, {expired_total} expired", end="")
    for h in HANDLERS:
        print("\nring wrap: " + census_line(h, paths[h]), end="")
    RAN.add("wrap")


# ---------------------------------------------------------------- 5. capacity boundaries
CAP = 2048


def place_all(pushes):
    """Physical offsets of the tasks of pushes made into an empty ring, one after another (no drain in between)."""
    m, offs = RingModel(1 << 26, 1 << 20), []
    for p in pushes:
        s = m.push([len(t.payload) for t in p])
        pos = s
        for t in p:
            offs.append(pos)
            pos += len(t.payload)
    return np.array(offs, np.int64)


def tune(pushes, var, make, t0, tt, metric, target, lo=FRAME, hi=6000):
    """Replace pushes[var[0]][var[1]] by make(L) for the first L that makes metric(tile_metrics of the tile of tasks
    [t0, t0 + tt), offsets, lengths) == target."""
    for L in range(lo, hi):
        pushes[var[0]][var[1]] = make(L)
        flat = [t for p in pushes for t in p]
        offs = place_all(pushes)
        lens = np.array([len(t.payload) for t in flat], np.int64)
        if metric(tile_metrics(offs[t0:t0 + tt], lens[t0:t0 + tt]), offs - offs[t0], lens[t0:]) == target:
            return pushes
    raise AssertionError(f"no length gives {target}")


def own_of_len(handler, L, seed=0):
    """A task of the handler's own shape of about / exactly L bytes."""
    if handler in ("identity", "crc32"):
        return string_task(max(L, FRAME))
    if handler == "json_sum":
        return json_task(L, seed)
    fpv = max(1, (L - FRAME) * 3 // 32)                 # base64 of 8 x fpv bytes: 4 ceil(8 fpv / 3) characters
    return tasks_of(synth.vadd_batch(1, floats_per_vec=fpv, seed=seed), "vadd")[0]


def boundary_cases(h):
    """-> [(case, pushes, indices of the tasks the case is about, the path the arithmetic predicts for them)]"""
    tt = TILE[h]
    avg = CAP // tt
    unstaged = "per-task" if h in ("crc32", "json_sum") else "global"
    cases = []
    # contiguous hull exactly CAP and CAP + 16: tile 1 of one push, starting misaligned behind tile 0
    for extra, want in ((0, "whole"), (16, unstaged)):
        tile0 = [own_of_len(h, 45 + 3 * j, j) for j in range(tt)]
        tile1 = [own_of_len(h, avg - 20, j) for j in range(tt)]
        p = tune([tile0 + tile1], (0, 2 * tt - 1), lambda L: string_task(L) if h == "vadd_f32" else own_of_len(h, L, 99),
                 tt, tt, lambda m, o, l: m[1] if m[0] else -1, CAP + extra, lo=40)
        cases.append((f"hull = in_cap + {extra}", p, list(range(tt, 2 * tt)), want))
    # scattered total exactly CAP and CAP + 16: tile 1 straddles two pushes
    for extra, want in ((0, "scattered"), (16, unstaged)):
        half = tt // 2
        p0 = [own_of_len(h, 40 + j, j) for j in range(tt)] + [own_of_len(h, avg - 45 + 3 * j, j) for j in range(half)]
        p1 = [own_of_len(h, avg - 45, j) for j in range(tt - half)] + [own_of_len(h, 60, j) for j in range(tt)]
        if sum(len(t.payload) for t in p0) % 256 == 0:
            p0[0] = own_of_len(h, len(p0[0].payload) + 1)
        p = tune([p0, p1], (1, tt - half - 1), lambda L: string_task(L) if h == "vadd_f32" else own_of_len(h, L, 98),
                 tt, tt, lambda m, o, l: -1 if m[0] else m[2], CAP + extra)
        cases.append((f"scattered = in_cap + {extra}", p, list(range(tt, 2 * tt)), want))
    if h in ("crc32", "json_sum"):
        # one task with mis + len + 16 exactly CAP and CAP + 1, in a tile that is too large to stage
        for extra, want in ((0, "per-task"), (1, "global")):
            small = own_of_len(h, 83 if h == "json_sum" else 37, 5)
            p = [[small, own_of_len(h, 1000), own_of_len(h, 300, 6), own_of_len(h, 90, 7)] + [own_of_len(h, 100, 8)] * 4]
            p = tune(p, (0, 1), lambda L: own_of_len(h, L, 4), 0, tt,
                     lambda m, o, l: -1 if m[1] <= CAP else int(o[1] & 15) + int(l[1]) + 16, CAP + extra, lo=1500)
            cases.append((f"mis + len + 16 = in_cap + {extra}", p, [1], want))
    # tiles of empty payloads only (inside a push, and a push of nothing else), and tiny tasks with a few over in_cap
    empties = [Task(b"", "str") for _ in range(2 * tt)]
    cases.append(("empty payloads", [[own_of_len(h, 61, 1)] * tt + empties + [own_of_len(h, 70, 2)] * tt, list(empties)], list(range(tt, 3 * tt)), "whole"))
    tiny = [own_of_len(h, 30 + (j % 40), j) if h != "json_sum" else json_task(80 + j % 40, j) for j in range(400)]
    for j in (37, 38, 200, 399):
        tiny[j] = own_of_len(h, CAP + 500 + j, j) if h != "vadd_f32" else string_task(CAP + 500 + j)
    cases.append(("tiny tasks, a few over in_cap", [tiny], [37, 38, 200, 399], "global"))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("h", HANDLERS)
def test_capacity_boundaries(stage, h):
    """Under in_cap = 2048: a contiguous tile whose hull is exactly in_cap and in_cap + 16, a scattered one whose per-task
    hulls add up to exactly in_cap and in_cap + 16, a single task with mis + len + 16 exactly in_cap and in_cap + 1,
    tiles of empty payloads only, and a window of tiny tasks with a few larger than in_cap."""
    q = stage(CAP)
    cases = boundary_cases(h)
    for name, pushes, idx, want in cases:
        for p in pushes:
            assert q.push([copy_task(t) for t in p])
        _, paths = q.drain_all(h)
        got = {paths[i] for i in idx}
        BOUNDARY.append((h, name, want, "/".join(sorted(got))))
        assert got == {want}, (h, name, got)
    RAN.add(f"boundary{h}")


# ---------------------------------------------------------------- 6. a peek leaves the ring as it was
@pytest.mark.gpu
@pytest.mark.parametrize("stage_bytes", [None, 16384])
def test_peek_leaves_the_ring_untouched(stage, stage_bytes):
    """vadd_f32's fast path rewrites the stage buffer in place and pickle-framed identity patches a frame header there:
    two peeks and then the real drain give the same records, equal to the oracle."""
    from oracle.pyoracle import funcloop
    q = stage(stage_bytes)
    rng = np.random.default_rng(61)
    for h, tasks in (("vadd_f32", tasks_of(synth.vadd_batch(3000, seed=8), "vadd") + tasks_of(synth.vadd_batch(700, floats_per_vec=5, seed=9), "vadd")),
                     ("identity", [Task(funcloop.frame_map_input("".join(chr(int(c)) for c in rng.integers(0x20, 0x7F, int(rng.integers(0, 400))))),
                                        "pickle", TF_PICKLE) for _ in range(2000)])):
        assert q.push(tasks)
        rs = [q.drain_all(h, peek=True)[0], q.drain_all(h, peek=True)[0]]
        r, paths = q.drain_all(h)
        rs.append(r)
        assert Counter(paths)["whole"] > 0
        recs = [x.records() for x in rs]
        assert recs[0] == recs[1] == recs[2]
    RAN.add(f"peek{stage_bytes}")


# ---------------------------------------------------------------- the census
@pytest.mark.gpu
def test_zz_census_reached_every_path():
    """Every (handler, path) pair the kernel has got at least CENSUS_FLOOR tasks over this file, and every capacity
    boundary case landed on the side the arithmetic predicts."""
    scenarios = {f"{name}{s}{h}" for h in HANDLERS for name, sizes in (("stage", STAGE_SIZES), ("across", (None, 16384, 49152)),
                                                                       ("partial", (None, 5120))) for s in sizes} \
        | {f"boundary{h}" for h in HANDLERS} | {"wrap"} | {f"peek{s}" for s in (None, 16384)}
    if not scenarios <= RAN:
        pytest.skip(f"the census needs the whole file; missing {sorted(scenarios - RAN)}")
    print("\ncensus (ready tasks by handler and path):")
    for h in HANDLERS:
        print("  " + " ".join(f"{p}={CENSUS[(h, p)]:6d}" for p in PATHS) + f"  {h}")
    print("capacity boundaries (handler, case, predicted, census):")
    for b in BOUNDARY:
        print("  " + " | ".join(b))
    low = {(h, p): CENSUS[(h, p)] for h in HANDLERS for p in KERNEL_PATHS[h] if CENSUS[(h, p)] < CENSUS_FLOOR}
    assert not low, low
    assert all(b[2] == b[3] for b in BOUNDARY)
