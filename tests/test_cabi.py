"""The C-ABI shared library loads on a CPU-only box and exports every symbol include/b200_train.h declares
(no compute calls here: those are the -m gpu tests)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "b200_train.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported_and_bound():
    from automodel_b200._lib import lib, SIGNATURES, LIB_PATH
    assert os.path.exists(LIB_PATH), "build with: python -c 'import __graft_entry__ as g; g.build()'"
    names = _declared()
    assert len(names) >= 30
    h = ctypes.CDLL(LIB_PATH)
    for n in names:
        assert hasattr(h, n), f"{n} declared in include/b200_train.h but not exported"
        assert n in SIGNATURES, f"{n} has no ctypes signature in automodel_b200/_lib.py"
    assert set(SIGNATURES) <= set(names), set(SIGNATURES) - set(names)
    assert lib().b200_abi_version() == 2


def test_errors_are_reported_not_raised():
    """Error behaviour of the ABI: negative code + message, no exception, no crash (CPU box: the device check must fail cleanly)."""
    import torch
    from automodel_b200._lib import lib
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    rc = lib().b200_device_check()
    assert rc < 0
    assert len(lib().b200_last_error()) > 0
    assert lib().b200_set_option(b"no_such_option", 1) == -1


def test_product_has_no_oracle_or_fallback_imports():
    """The shipped package must not import the oracle, the CPU stand-in kernels or torch matmul paths."""
    pkg = os.path.join(ROOT, "automodel_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "import oracle" not in src and "from oracle" not in src, fn
            assert "cpu_kernels" not in src, fn


def test_header_is_plain_c_and_binds_from_a_c_program(tmp_path):
    """include/b200_train.h is the boundary a non-Python host would bind (cgo / JNI / dlopen): it must compile as C99 on its own, and
    a C program linked against libb200_train.so must be able to call it (no compute here: error path + option table + version)."""
    import shutil
    import subprocess
    from automodel_b200._lib import LIB_PATH
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    inc = os.path.join(ROOT, "include")
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-x", "c", os.path.join(inc, "b200_train.h")], check=True)
    src = tmp_path / "smoke.c"
    src.write_text(r'''
#include <stdio.h>
#include <string.h>
#include "b200_train.h"
int main(void) {
  if (b200_abi_version() != 2) return 1;
  if (b200_set_option("gemm_sched", 0) != 0) return 2;
  if (b200_set_option("no_such_option", 1) >= 0) return 3;
  if (strlen(b200_last_error()) == 0) return 4;
  /* argument validation happens before any device work */
  if (b200_gemm_bf16(B200_GEMM_NT, 0, 0, 0, 0, 0, 0, 0, 0, /*M*/ 0, 16, 16, 0, 0, 0, 0) >= 0) return 5;
  printf("abi %d ok: %s\n", b200_abi_version(), b200_last_error());
  return 0;
}
''')
    exe = tmp_path / "smoke"
    libdir = os.path.dirname(LIB_PATH)
    subprocess.run([gcc, "-std=c99", "-Wall", "-I", inc, str(src), "-o", str(exe), "-L", libdir, "-lb200_train", f"-Wl,-rpath,{libdir}"], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert "abi 2 ok" in r.stdout
