"""Runs one joint_rnnt_loss forward+backward on the tensor-core path and saves costs + gradients to an .npz.
Used by tests that compare two PROCESS-level configurations of the library (environment switches are read once per
process), e.g. the multi-chunk backward (RNNTB200_CHUNK_MB) against the single-chunk one.

    python tools/joint_dump.py OUT.npz B T U V H seed ragged keep [bound]
    python tools/joint_dump.py OUT.npz --inputs IN.npz keep [bound]

The first form runs synthetic inputs (tests/test_gpu_joint.py: synth).  The second runs the arrays of IN.npz: enc,
pred, W, b, labels, input_lengths, label_lengths and blank as synth() returns them, and optionally `scale`, the upstream
gradient of each utterance's cost (default 1/B).
bound: 0 = none, 1 = pass valid_tiles = valid_tile_count(host lengths), N > 1 = pass valid_tiles = N (a deliberately wrong promise).
The .npz also records which forward kernels ran ("kernels"), so that a test can tell keep mode from the recomputing mode.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

if __name__ == "__main__":
    from test_gpu_joint import run_joint, synth
    out = sys.argv[1]
    if sys.argv[2] == "--inputs":
        k = dict(np.load(sys.argv[3]))
        rest = sys.argv[4:]
    else:
        B, T, U, V, H, seed, ragged = (int(x) for x in sys.argv[2:9])
        k = synth(B, T, U, V, H, seed, bool(ragged))
        rest = sys.argv[9:]
    keep = int(rest[0])
    bound = int(rest[1]) if len(rest) > 1 else 0
    scale = k.pop("scale", None)
    import rnnt_speech_recognition_b200 as rb
    from rnnt_speech_recognition_b200 import _lib
    vt = None if bound == 0 else (rb.valid_tile_count(k["input_lengths"], k["label_lengths"]) if bound == 1 else bound)
    _lib.set_timing(True)
    costs, grads = run_joint(k, "bf16", scale=scale, keep=bool(keep), valid_tiles=vt)
    names = sorted({n for n, _ in _lib.get_timings()})
    np.savez(out, costs=costs, d_enc=grads[0], d_pred=grads[1], dW=grads[2], db=grads[3], kernels=np.array(names))
