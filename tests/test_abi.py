"""CPU checks of the drop-in boundary: the C-ABI library loads and exports every symbol include/a2f.h declares,
and the ctypes binding covers each of them.  No compute call is made (no GPU here)."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "a2f.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"\b(a2f_[a-z0-9_]+)\s*\(", src)
    return sorted(set(names))


def test_header_symbols_exported(a2f_lib):
    names = _declared()
    assert len(names) >= 20
    missing = [n for n in names if not hasattr(a2f_lib, n)]
    assert not missing, f"declared in include/a2f.h but not exported: {missing}"


def test_header_is_plain_c():
    """The boundary is a C ABI: include/a2f.h must compile as C (a declaration that slipped inside a struct body would
    still be valid C++, and did go unnoticed once)."""
    import shutil
    import subprocess

    gcc = shutil.which("gcc")
    if gcc is None:
        import pytest
        pytest.skip("no gcc")
    r = subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-x", "c", os.path.join(ROOT, "include", "a2f.h")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_binding_covers_header():
    import a2f_b200

    names = _declared()
    unbound = [n for n in names if n not in a2f_b200.lib._SIGNATURES]
    assert not unbound, f"no ctypes signature for: {unbound}"
    extra = [n for n in a2f_b200.lib._SIGNATURES if n not in names]
    assert not extra, f"bound but not declared in the header: {extra}"


def test_version_and_status_strings(a2f_lib):
    assert a2f_lib.a2f_version() == 100
    assert b"A2F_OK" in a2f_lib.a2f_status_string(0)
    assert b"sm_100" in a2f_lib.a2f_status_string(-2)


_NO_GPU_CHILD = """
import ctypes as C
import a2f_b200
L = a2f_b200.lib
rc = L.load().a2f_gemm(C.byref(L.GemmArgs()), 0, None)
assert rc != 0, rc
try:
    L.check(rc, "a2f_gemm")
except a2f_b200.A2FError:
    print("A2F_REFUSED")
"""


def test_compute_fails_loudly_without_gpu(a2f_lib):
    """No silent fallback: without a CUDA device a compute entry point must return an error status.  Checked in a child
    process that sees no device (CUDA_VISIBLE_DEVICES=""), so that it runs on GPU machines too."""
    import subprocess
    import sys

    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", _NO_GPU_CHILD], cwd=ROOT, env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "A2F_REFUSED" in r.stdout, r.stdout + r.stderr


def test_modules_refuse_cpu_tensors():
    import pytest
    import torch
    import a2f_b200
    from a2f_b200 import modules

    m = modules.Voca(15069, 12)
    with pytest.raises(a2f_b200.A2FError):
        m(torch.zeros(2, 29, 16), torch.zeros(2, 12), torch.zeros(2, 5023, 3))
