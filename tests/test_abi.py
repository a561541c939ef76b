"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol that
include/rnnt_b200.h declares, and its pure / argument-checking entry points behave like the
reference's (rnnt_entrypoint.cpp:14-35, 49-60, 96-128).  No compute call needs a GPU here."""
import ctypes as C
import json
import os
import re

import pytest

from conftest import ROOT


@pytest.fixture(scope="module")
def L():
    from rnnt_speech_recognition_b200 import _lib
    return _lib.load()


def reference_abi():
    """What the reference's rnnt.h and library define at the boundary (tests/golden/make_golden.py: reference_abi)."""
    with open(os.path.join(ROOT, "tests", "golden", "reference_abi.json")) as f:
        return json.load(f)


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "rnnt_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"^\s*(?:rnntStatus_t|int|void|const char\*|unsigned long long)\s+(\w+)\s*\(", src, flags=re.M)
    return sorted(set(names))


def test_exports_every_declared_symbol(L):
    from rnnt_speech_recognition_b200 import _lib
    names = declared_symbols()
    assert set(names) == set(_lib.EXPORTS), (names, _lib.EXPORTS)
    for n in names:
        assert getattr(L, n) is not None


def test_version_and_status_strings(L):
    assert L.get_warprnnt_version() == 1
    want = ["no error", "cuda memcpy or memset failed", "invalid value", "execution failed", "unknown error"]
    for i, w in enumerate(want):
        assert L.rnntGetStatusString(i).decode() == w
    assert L.rnntGetStatusString(17).decode() == "unknown error"
    ref = reference_abi()            # identical to the unmodified reference library
    assert L.get_warprnnt_version() == ref["version"]
    assert [L.rnntGetStatusString(i).decode() for i in range(6)] == ref["status_strings"]


def test_workspace_size(L, oracle):
    s = C.c_size_t(0)
    assert L.get_workspace_size(0, 3, 2, True, C.byref(s), 4) == 2       # INVALID_VALUE, rnnt_entrypoint.cpp:102-105
    assert L.get_workspace_size(4, 3, -1, False, C.byref(s), 4) == 2
    for (T, U, B) in ((4, 3, 2), (512, 128, 32), (1600, 200, 64)):
        assert L.get_workspace_size(T, U, B, False, C.byref(s), 4) == 0
        assert (0, s.value) == oracle.get_workspace_size(T, U, B, False)  # reference CPU figure
        assert L.get_workspace_size(T, U, B, True, C.byref(s), 4) == 0
        SK = (T + U - 1) * U
        assert s.value == B * (4 * SK + T * U + 2) * 4
        assert s.value >= oracle.get_workspace_size(T, U, B, True)[1]    # never smaller than the reference's


def test_argument_checks_without_gpu(L):
    from rnnt_speech_recognition_b200 import _lib
    opt = _lib.RnntOptions(_lib.RNNT_GPU, 0, None, 0, 4, 3, True)
    one = C.c_void_p(16)  # never dereferenced: every call below must bail out in the argument checks
    assert L.compute_rnnt_loss(None, None, one, one, one, 5, 1, one, one, opt) == 2
    assert L.compute_rnnt_loss(one, None, one, one, one, 0, 1, one, one, opt) == 2
    assert L.compute_rnnt_loss(one, None, one, one, one, 5, 0, one, one, opt) == 2
    assert L.compute_rnnt_loss_fp64(one, None, one, one, one, 5, 1, None, one, opt) == 2
    bad = _lib.RnntOptions(_lib.RNNT_GPU, 0, None, 0, 0, 3, True)
    assert L.compute_rnnt_loss(one, None, one, one, one, 5, 1, one, one, bad) == 2
    cpu = _lib.RnntOptions(_lib.RNNT_CPU, 1, None, 0, 4, 3, True)
    assert L.compute_rnnt_loss(one, None, one, one, one, 5, 1, one, one, cpu) == 3   # no CPU fallback
    d = _lib.JointDesc(2, 4, 3, 64, 0, 0, 0, None)
    s = C.c_size_t(0)
    assert L.rnntb200_joint_workspace_size(C.byref(d), C.byref(s)) == 2
    d = _lib.JointDesc(2, 4, 3, 64, 128, 0, 0, None)
    assert L.rnntb200_joint_workspace_size(C.byref(d), C.byref(s)) == 0 and s.value > 0
    assert L.rnntb200_joint_loss_forward(C.byref(d), None, one, one, one, one, one, one, one, one) == 2


def test_struct_layout_matches_reference_header():
    from rnnt_speech_recognition_b200 import _lib
    assert C.sizeof(_lib.RnntOptions) == 32            # rnnt.h:43-64 on x86-64
    assert _lib.RnntOptions.stream.offset == 8 and _lib.RnntOptions.blank_label.offset == 16
    assert _lib.RnntOptions.batch_first.offset == 28


def test_reference_header_links_against_this_library():
    """Header-level ABI check: tests/abi_harness/abi_harness.cpp uses the warp-transducer API through include/rnnt_b200.h
    and is linked against librnnt_b200.so -- what tensorflow_binding/src/warprnnt_op.cc:105-141 and
    pytorch_binding/src/binding.cpp:84-154 do.  The rnntOptions layout and enum values it sees are those the same
    harness sees through the reference's own rnnt.h, and every function rnnt.h declares is declared here and exported.
    `link` mode resolves every symbol and exercises the host-only entry points; the known-answer run on a GPU is
    tests/test_gpu_loss_op.py::test_abi_harness_kat."""
    import subprocess
    import sys
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge
    from rnnt_speech_recognition_b200 import _lib
    L = _lib.load()
    ref = reference_abi()
    assert set(ref["header_functions"]) <= set(declared_symbols())
    for n in ref["header_functions"]:
        assert getattr(L, n) is not None
    exe = ge.build_abi_harness()
    r = subprocess.run([exe, "layout"], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stdout + r.stderr
    assert json.loads(r.stdout) == ref["layout"]
    r = subprocess.run([exe, "link"], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "link ok" in r.stdout
