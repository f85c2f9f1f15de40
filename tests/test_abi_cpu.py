"""CPU-side checks of the drop-in boundary: the C-ABI library loads without a GPU and exports every
function include/dyros_b200.h declares; the ctypes mirror covers exactly that set."""
import ctypes
import os
import subprocess
import sys

import pytest

from isaacgymdyros_b200 import native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.isfile(native.LIB_PATH):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "isaacgymdyros_b200", "csrc")], stdout=subprocess.DEVNULL)
    return native.load()


def test_header_symbols_all_exported(lib):
    syms = native.header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/dyros_b200.h but not exported"
    assert sorted(native.SIGNATURES) == syms, "ctypes SIGNATURES and the header disagree"


def test_abi_version_and_error_string(lib):
    assert lib.dyros_abi_version() == native.ABI_VERSION == 3
    # NULL handles are rejected with a message and no CUDA call
    assert lib.dyros_simulate(None, 0, None) != 0
    assert b"sim is NULL" in lib.dyros_last_error()
    assert lib.dyros_task_step(None, None, None) != 0
    assert b"task is NULL" in lib.dyros_last_error()
    assert lib.dyros_sim_destroy(None) == 0 and lib.dyros_task_destroy(None) == 0


def test_struct_layouts_match_header_sizes(lib):
    # pointer-only structs: one pointer per declared member
    assert ctypes.sizeof(native.DyrosSimBuffers) == 8 * len(native.SIM_BUFFERS)
    assert ctypes.sizeof(native.DyrosTaskBuffers) == 8 * (len(native.TASK_BUFFERS) + len(native.TASK_SHARED) + len(native.TASK_OPTIONAL))
    assert ctypes.sizeof(native.DyrosNoiseInjection) == 8 * len(native.NOISE_FIELDS)
    # compile a tiny C program against the header and compare sizeof() of the mixed structs
    src = r'''
#include <stdio.h>
#include "dyros_b200.h"
int main(void){printf("%zu %zu %zu %zu %zu %zu\n", sizeof(DyrosModelDesc), sizeof(DyrosSimDesc), sizeof(DyrosSimBuffers),
  sizeof(DyrosTaskBuffers), sizeof(DyrosTaskDesc), sizeof(DyrosNoiseInjection)); return 0;}
'''
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "s.c"), "-o", os.path.join(d, "s")])
        out = subprocess.check_output([os.path.join(d, "s")]).decode().split()
    want = [ctypes.sizeof(x) for x in (native.DyrosModelDesc, native.DyrosSimDesc, native.DyrosSimBuffers,
                                       native.DyrosTaskBuffers, native.DyrosTaskDesc, native.DyrosNoiseInjection)]
    assert [int(x) for x in out] == want


def test_core_refuses_to_run_without_gpu():
    """In a child process with every CUDA device hidden, so that it runs on GPU machines too."""
    code = ("import pytest\nfrom isaacgymdyros_b200 import native\nfrom isaacgymdyros_b200.core import DyrosCore\n"
            "with pytest.raises(native.DyrosError):\n    DyrosCore(4)\n")
    subprocess.run([sys.executable, "-c", code], cwd=ROOT, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, check=True)


def test_header_is_plain_c(tmp_path):
    """include/dyros_b200.h is the drop-in boundary for C callers (cgo / JNI / ctypes generators): it must compile as C11 by
    itself, with nothing but its own includes."""
    import os
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        import pytest
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "hdr.c"
    src.write_text('#include "dyros_b200.h"\nint main(void) { return sizeof(DyrosPpoPeers) > 0 && sizeof(DyrosModelDesc) > 0 ? 0 : 1; }\n')
    subprocess.check_call(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(root, "include"), "-fsyntax-only", str(src)])
