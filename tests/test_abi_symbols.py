"""CPU-side checks of the drop-in boundary: the library builds, loads, and exports exactly the
symbols include/b9gpu.h declares; host-only helpers match the reference's known answers."""
import os
import re
import subprocess

import pytest

from beta9_b200 import _lib as L
from beta9_b200 import build as B
from beta9_b200.device_queue import task_queue_scale
from tests.test_oracle_reference_answers import AUTOSCALER_CASES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def so_path():
    return B.build()


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "b9gpu.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(b9_[a-z0-9_]+)\s*\(", txt)))


def test_header_and_binding_agree():
    assert header_symbols() == sorted(L.SYMBOLS)


def test_library_exports_every_declared_symbol(so_path):
    out = subprocess.check_output(["nm", "-D", "--defined-only", so_path], text=True)
    exported = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    missing = [s for s in header_symbols() if s not in exported]
    assert not missing, missing
    # and nothing b9_* is exported that the header does not declare
    extra = sorted(s for s in exported if s.startswith("b9_") and s not in header_symbols())
    assert not extra, extra


def test_library_loads_and_reports_abi(so_path):
    lib = L.load()
    assert lib.b9_abi_version() == 2
    assert lib.b9_handler_name(0) == b"identity" and lib.b9_handler_name(3) == b"json_sum"
    assert lib.b9_handler_name(99) is None
    assert lib.b9_handler_id(b"crc32") == 1 and lib.b9_handler_id(b"echo") == 0
    assert lib.b9_handler_id(b"nope") == L.B9_ENOSYS


def test_sass_is_sm100a(so_path):
    out = subprocess.run(["cuobjdump", "-lelf", so_path], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out


@pytest.mark.parametrize("q,tpc,mc,mr,desired,valid", AUTOSCALER_CASES)
def test_scale_func_known_answers_through_abi(so_path, q, tpc, mc, mr, desired, valid):
    # pkg/abstractions/taskqueue/autoscaler_test.go:34-123
    assert task_queue_scale(q, tpc, mc, mr) == (desired, valid)


def test_no_device_fails_loudly(so_path):
    """In a process that sees no CUDA device (CUDA_VISIBLE_DEVICES="" hides those of a GPU machine), creating a
    queue raises B9_ENODEV with the "no CPU path" message."""
    import sys
    code = ("from beta9_b200 import _lib as L\n"
            "from beta9_b200.device_queue import DeviceQueue\n"
            "assert L.load().b9_device_count() == 0\n"
            "try:\n"
            "    DeviceQueue()\n"
            "except L.B9Error as e:\n"
            "    assert e.code == L.B9_ENODEV and 'no CPU path' in str(e), (e.code, str(e))\n"
            "else:\n"
            "    raise AssertionError('DeviceQueue() without a device did not raise')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=120,
                       env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
    assert r.returncode == 0, r.stderr[-2000:]


def test_header_is_plain_c99_and_the_c_example_links(so_path, tmp_path):
    """include/b9gpu.h must be usable from C (cgo compiles it as C): examples/c_api_demo.c under -std=c99 -pedantic
    -Werror, then linked against the library. Without a GPU the program must stop at b9_ctx_create with the
    "no CPU path" message; with one it prints three records."""
    import shutil
    import subprocess
    cc = shutil.which("gcc") or shutil.which("cc")
    if not cc:
        pytest.skip("no C compiler")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = os.path.join(root, "examples", "c_api_demo.c")
    inc = os.path.join(root, "include")
    r = subprocess.run([cc, "-std=c99", "-pedantic", "-Wall", "-Werror", "-fsyntax-only", "-I" + inc, src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    exe = str(tmp_path / "c_api_demo")
    libdir = os.path.dirname(so_path)
    r = subprocess.run([cc, "-std=c99", "-I" + inc, src, "-L" + libdir, "-lb9gpu", "-Wl,-rpath," + libdir, "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    if r.returncode != 0:
        assert "no CPU path" in r.stderr, r.stderr               # CPU-only host: fails loudly, as designed
    else:
        assert "hello" in r.stdout and "from an HTTP body" in r.stdout and "caf\\u00e9" in r.stdout, r.stdout
