"""Workspace of the tensor-core path at any (H, V) -- a pure function of the descriptor, so no GPU is needed."""
import ctypes as C

import numpy as np
import pytest

import rnnt_speech_recognition_b200 as rb
from rnnt_speech_recognition_b200 import _lib


def workspace(B, T, U, H, V, keep=0, bound=0, precision=1):
    L = _lib.load(build_if_missing=True)
    d = _lib.JointDesc(B, T, U, H, V, 0, precision, None, bound, keep)
    s = C.c_size_t(0)
    st = L.rnntb200_joint_workspace_size(C.byref(d), C.byref(s))
    return st, s.value


def c5_bound():
    rng = np.random.default_rng(0)
    il, ll = rng.integers(100, 1601, 64), rng.integers(10, 201, 64) - 1
    return rb.valid_tile_count(il, ll)


def test_aligned_workspace_sizes_are_unchanged():
    """The sizes the library returned before any vocabulary / joint width became legal (BASELINE C2, C3 in keep mode, C5
    with and without a valid-tile bound): aligned descriptors keep exactly their layout."""
    assert c5_bound() == 48415
    assert workspace(16, 256, 64, 320, 256) == (0, 176100864)
    assert workspace(32, 512, 128, 640, 1024, keep=1) == (0, 4732076544)
    assert workspace(64, 1600, 200, 640, 4096, keep=1) == (0, 16543908608)
    assert workspace(64, 1600, 200, 640, 4096, keep=1, bound=48415) == (0, 54589372160)


def staged_bytes(B, T, U, Hp):
    a = lambda n: (n + 255) // 256 * 256
    return 2 * a(B * T * Hp * 4) + a(B * U * Hp * 4)


@pytest.mark.parametrize("B,T,U,H,V,keep,bound", [
    (32, 512, 128, 640, 1025, 1, 0),     # V only: no staged arrays
    (4, 200, 64, 640, 4073, 1, 0),
    (8, 256, 96, 640, 31, 0, 0),
    (32, 512, 128, 600, 1024, 1, 0),     # H only
    (3, 25, 11, 50, 33, 1, 0),
    (2, 18, 7, 1, 100, 0, 0),
    (2, 19, 9, 767, 130, 1, 0),
    (64, 1600, 200, 600, 4073, 1, 48415),
])
def test_unaligned_workspace_is_the_padded_one_plus_the_staged_rows(B, T, U, H, V, keep, bound):
    Hp, Vp = (H + 63) // 64 * 64, (V + 63) // 64 * 64
    st, got = workspace(B, T, U, H, V, keep, bound)
    assert st == 0
    st, padded = workspace(B, T, U, Hp, Vp, keep, bound)
    assert st == 0
    assert got == padded + (staged_bytes(B, T, U, Hp) if H != Hp else 0)

