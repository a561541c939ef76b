"""Tensor-core joint loss at extreme logit gaps, against the fp64 oracle.

The forward epilogue takes every softmax numerator of a lattice row against one frame: the maximum of the row's first
32 logits, moved up when a later 32-column group reaches 2^64 against it.  The backward scales the kept numerators by a
per-row factor that is flushed to 0 below 1e-30.  Rows whose maximum lies far beyond their first 32 columns (a confident
prediction of a token past column 31) exercise the frame switch; if the kept numerators were not taken against the
row's final frame, such rows would lose their gradient while the costs stayed right.

Every input here gives one dominant column v* a logit `gap` nats above the rest, built so that 16-bit operand rounding
stays out of the way:
  * "bias": the gap is on b[v*] (fp32 in the epilogue, exact); every row is extreme.
  * "row":  one hidden unit h0 with enc[..., h0] = +-20 on alternate time steps and pred[..., h0] = 0, so z = +-1 after
            tanh and fp16; W[h0, v*] = gap (exact in fp16) and the rest of W's row h0 is zero.  Half the rows of every
            16 x 8 lattice tile are extreme (v* at +gap), the other half ordinary (v* at -gap).
The four utterances of a batch carry the upstream gradients 1, 1/32, -0.5 and 1e-4; the per-utterance gradients are
checked one utterance at a time, so a small scale cannot hide behind a large one.

The same inputs through the fp32 joint path and through the loss op on the oracle's materialised logits (both take the
true row maximum) pin that the inputs themselves are well posed."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, assert_close, fp32_tol
from test_gpu_joint import dev, run_joint, synth
from test_gpu_joint_bf16 import NAMES, TC_COST_RTOL, TC_GRAD_NTOL, oracle_of

pytestmark = pytest.mark.gpu

GS = np.array([1.0, 1.0 / 32, -0.5, 1e-4])       # upstream gradient of each utterance's cost
GAPS = [0, 40, 60, 66, 70, 100, 150]              # nats; 2^64 is 44.4 nats, the flush threshold 1e-30 is 69 nats
TC_FROB = 5e-3


def dominant(V, where):
    """(v*, blank) of a case.  'wrong': a class that is never the label; 'label': every label is v*; 'blank': v* is the
    blank; 'first32': a wrong class inside the first 32 columns, where the frame is the true row maximum (control)."""
    if where == "wrong":
        return V - 1, 0           # the last column: alone in the last 32-column group of V = 4097, in a partial group of V = 1000
    if where == "label":
        return min(40, V - 1), 0  # second 32-column group (V >= 41)
    if where == "blank":
        return V - 1, V - 1
    assert where == "first32"
    return 7, 0


def extreme(V, H, gap, where, form, seed=0, B=4, T=20, U=9):
    k = synth(B, T, U, V, H, seed, ragged=True)
    vs, blank = dominant(V, where)
    rng = np.random.default_rng(seed + 1000)
    if where == "label":
        k["labels"][:] = vs
    else:
        cand = np.array([v for v in range(V) if v not in (vs, blank)])
        k["labels"] = rng.choice(cand, size=k["labels"].shape).astype(np.int32)
    k["blank"] = np.int32(blank)
    if form == "bias":
        k["b"][vs] += np.float32(gap)
    else:
        h0 = H - 1
        k["enc"][:, :, h0] = np.where(np.arange(T) % 2 == 0, 20.0, -20.0).astype(np.float32)
        k["pred"][:, :, h0] = 0.0
        k["W"][h0, :] = 0.0
        k["W"][h0, vs] = np.float32(gap)
    return k


def check_tc(oracle, k, keep):
    o = oracle_of(oracle, k, GS, int(k["blank"]))
    costs, grads = run_joint(k, "bf16", scale=GS, keep=keep)
    check_vs_oracle(k, costs, grads, o)


def check_vs_oracle(k, costs, grads, o):
    """16-bit tolerances of test_gpu_joint_bf16.py; d_enc / d_pred per utterance, dW / db over the batch."""
    assert_close(costs, o["costs"], rtol=TC_COST_RTOL, atol=1e-3, what="costs")

    def close(got, want, what):
        assert_close(got, want, rtol=0, atol=0, ntol=TC_GRAD_NTOL, what=what)
        rel = np.linalg.norm(got - want) / np.linalg.norm(want)
        assert rel < TC_FROB, (what, rel)

    for g, n in zip(grads, NAMES):
        if n in ("d_enc", "d_pred"):
            for b in range(len(GS)):
                close(g[b], o[n][b], "%s[utterance %d, scale %g]" % (n, b, GS[b]))
        else:
            close(g, o[n], n)


@pytest.mark.parametrize("keep", [True, False])   # backward from the kept numerators / after re-running the projection
@pytest.mark.parametrize("gap", GAPS)
@pytest.mark.parametrize("where", ["wrong", "label", "blank", "first32"])
@pytest.mark.parametrize("form", ["bias", "row"])
def test_extreme_gap_vs_oracle(oracle, form, where, gap, keep):
    """V = 128, H = 64: every dominant-column role at every gap."""
    check_tc(oracle, extreme(128, 64, gap, where, form), keep)


@pytest.mark.parametrize("keep", [True, False])
@pytest.mark.parametrize("gap", [0, 66, 150])
@pytest.mark.parametrize("form", ["bias", "row"])
@pytest.mark.parametrize("V,H,where", [
    (31, 64, "wrong"),       # one 32-column group: the frame is always the true maximum (control)
    (31, 50, "label"),       # ... with an unaligned joint width
    (128, 50, "wrong"),      # h0 = 49: the last real hidden unit before the padding
    (1000, 64, "wrong"),     # v* = 999 in the partial last group
    (1000, 50, "label"),
    (4097, 64, "blank"),     # Vp > 4096: the bias comes from global memory; blank = 4096 alone in the last group
    (4097, 50, "wrong"),
])
def test_extreme_gap_shapes(oracle, V, H, where, form, gap, keep):
    check_tc(oracle, extreme(V, H, gap, where, form, seed=V + H), keep)


@pytest.mark.parametrize("gap", GAPS)
@pytest.mark.parametrize("where", ["wrong", "label", "blank", "first32"])
@pytest.mark.parametrize("form", ["bias", "row"])
def test_extreme_gap_fp32_controls(oracle, form, where, gap):
    """The fp32 joint path and the loss op on materialised logits, at their own (fp32) tolerances, on the same inputs."""
    import rnnt_speech_recognition_b200 as rb
    k = extreme(128, 64, gap, where, form)
    blank = int(k["blank"])
    o = oracle_of(oracle, k, GS, blank)
    costs, grads = run_joint(k, "fp32", scale=GS)
    assert_close(costs, o["costs"], rtol=1e-5, atol=1e-4, what="fp32 costs")
    # fp32 exponents of magnitude |cost| carry eps32 * |cost| of round-off (test_c2_full_size_vs_oracle)
    cmax = float(np.abs(o["costs"]).max())
    for g, n in zip(grads, NAMES):
        assert_close(g, o[n], rtol=1e-4, atol=1e-6, ntol=max(1e-5, 2e-7 * cmax), what="fp32 " + n)
    # loss op on the oracle's logits (rounded to fp32, the op's input type)
    x = oracle.joint_forward(*(k[n].astype(np.float64) for n in ("enc", "pred", "W", "b"))).astype(np.float32)
    oc, og = oracle.rnnt_logits_grad(x.astype(np.float64), k["labels"], k["input_lengths"], k["label_lengths"], blank)
    acts = dev(x).requires_grad_()
    c = rb.rnnt_loss(acts, dev(k["labels"], torch.int32), dev(k["input_lengths"], torch.int32),
                     dev(k["label_lengths"], torch.int32), blank)
    (c * dev(GS, torch.float32)).sum().backward()
    assert_close(c.detach().cpu().numpy(), oc, rtol=1e-5, atol=1e-4, what="op costs")
    assert_close(acts.grad.cpu().numpy(), og * GS[:, None, None, None], what="op logit grads", **fp32_tol(oc))


@pytest.mark.parametrize("keep", ["1", "0"])
def test_extreme_gap_one_cta_kernels(oracle, tmp_path, keep):
    """The one-CTA kernel forms (RNNTB200_FWD=3 RNNTB200_DZ=1 RNNTB200_DW=1, selected once per process, hence the child
    process): their forward epilogue is a separate copy of the frame logic."""
    k = extreme(1000, 64, 100, "wrong", "bias")
    inp, out = str(tmp_path / "in.npz"), str(tmp_path / "out.npz")
    np.savez(inp, scale=GS, **k)
    env = dict(os.environ, RNNTB200_FWD="3", RNNTB200_DZ="1", RNNTB200_DW="1")
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "joint_dump.py"), out, "--inputs", inp, keep],
                   check=True, env=env, timeout=300)
    r = dict(np.load(out))
    kernels = " ".join(str(x) for x in r["kernels"])
    assert "joint_tc3_kernel" in kernels and "joint_tc4_kernel" not in kernels and "bwd_dw2_kernel" not in kernels
    check_vs_oracle(k, r["costs"], [r[n] for n in NAMES], oracle_of(oracle, k, GS, int(k["blank"])))
