"""Tensor-core path (tcgen05 fused joint kernels: fp16 forward projection, own bf16 dZ / dW gradient GEMMs) against the
fp64 oracle -- small shapes, BASELINE C2 at FULL size, and one full BASELINE C3 utterance -- and against the fp32 exact
CUDA path.  16-bit operands carry 2^-12 (forward) / 2^-9 (gradient GEMMs) relative rounding, so this path is held to
its own measured tolerance (DESIGN.md "Tolerances"), not to the fp32 rtol 1e-4 gate."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, assert_close
from test_gpu_joint import run_joint, synth

pytestmark = pytest.mark.gpu

TC_COST_RTOL = 2e-4       # measured <= 4e-5 (profiles/r02/accuracy.json)
TC_GRAD_NTOL = 1e-2       # element-wise: |err| <= ntol * max|grad| (bf16 gradient operands, 2^-9 each); Frobenius checks use 5e-3
NAMES = ("d_enc", "d_pred", "dW", "db")


def oracle_of(oracle, k, gs, blank=0):
    return oracle.joint_loss_grad(*(k[n].astype(np.float64) for n in ("enc", "pred", "W", "b")), k["labels"],
                                  k["input_lengths"], k["label_lengths"], blank, grad_scale=gs)


@pytest.mark.parametrize("B,T,U,V,H,seed,ragged", [
    (2, 20, 8, 64, 64, 0, False),        # one tile per utterance row, single K block, single V chunk, single-block dW items
    (3, 37, 19, 128, 128, 1, True),      # ragged, partially filled tiles
    (2, 50, 40, 192, 320, 2, True),      # V chunk of 64 x3, 5 K blocks, one dZ pass of 320 columns (shared TMEM zone)
    (1, 9, 140, 64, 64, 3, False),       # U > 128: 18 u-blocks per t-block
    (2, 33, 128, 512, 640, 4, True),     # H = 640: two dZ passes, double + single dW items, two v-tiles
    (2, 40, 24, 320, 768, 6, True),      # H = 768 (largest supported), V = 320: a 64-wide last v-tile
    # every accumulator plan of the dZ kernel and every block-slot layout of the dW kernel (H), partial last v-tiles (V)
    (2, 24, 12, 576, 256, 7, True),      # H = 256: one pass, no shared zone; dW blocks [0, 1, SCALE]: a (SCALE, empty) pair; V = 512 + 64
    (1, 20, 10, 1088, 512, 8, False),    # H = 512: two passes of 256 columns; three dW v-tiles (512, 512, 64)
    (2, 18, 9, 128, 448, 9, True),       # H = 448: two passes of 224 columns (7 chunks over 4 epilogue groups)
    (2, 18, 9, 256, 576, 10, True),      # H = 576: shared zone of 64 columns -- two epilogue groups own no shared chunk
    (1, 17, 20, 192, 384, 11, False),    # H = 384: one pass, shared zone of 256 columns, private 128
    (2, 10, 5, 64, 192, 12, True),       # H = 192: six chunks, 1.5 dW blocks
    (1, 16, 8, 640, 704, 13, False),     # H = 704: two passes of 352 columns, shared zone 192
])
@pytest.mark.parametrize("keep", [True, False])   # backward from the kept numerators / after re-running the projection
def test_tc_vs_oracle(oracle, B, T, U, V, H, seed, ragged, keep):
    k = synth(B, T, U, V, H, seed, ragged)
    gs = np.linspace(0.5, 1.5, B)
    o = oracle_of(oracle, k, gs)
    costs, grads = run_joint(k, "bf16", scale=gs, keep=keep)
    assert_close(costs, o["costs"], rtol=TC_COST_RTOL, atol=1e-3, what="costs")
    for g, n in zip(grads, NAMES):
        assert_close(g, o[n], rtol=0, atol=0, ntol=TC_GRAD_NTOL, what=n)
    # padded positions of d_enc / d_pred are exactly zero
    for b in range(B):
        assert not grads[0][b, k["input_lengths"][b]:].any()
        assert not grads[1][b, k["label_lengths"][b] + 1:].any()


def test_c2_full_size_vs_oracle(oracle):
    """BASELINE C2 (B=16 T=256 U=64 V=256 H=320) at full size: the fp32 exact path at the north-star tolerance and the
    tensor-core path at its own, both against the fp64 oracle (seconds on the host cores)."""
    k = synth(16, 256, 64, 256, 320, 5, ragged=True)
    gs = np.full(16, 1.0 / 16)
    o = oracle_of(oracle, k, gs)
    c32, g32 = run_joint(k, "fp32")
    assert_close(c32, o["costs"], rtol=1e-5, atol=1e-3, what="fp32 costs")
    # fp32 arithmetic on exponents of magnitude |cost| ~ 1.5e3 carries eps32 * |cost| ~ 1e-4 of relative round-off per
    # cell (conftest.fp32_tol: the unmodified reference in fp32 is itself that far from its fp64 run): the north-star
    # rtol 1e-4 is met on the costs; gradients get the cost-scaled norm-wise floor
    cmax = float(np.abs(o["costs"]).max())
    for g, n in zip(g32, NAMES):
        rel = np.linalg.norm(g - o[n]) / np.linalg.norm(o[n])
        assert rel < 3e-4, ("fp32 " + n, rel)     # measured 1.4e-4: alpha, beta ~ 1.5e3 are stored in fp32 (ulp 1.2e-4)
        assert_close(g, o[n], rtol=1e-4, atol=1e-6, ntol=max(2e-5, 2e-7 * cmax), what="fp32 " + n)
    c16, g16 = run_joint(k, "bf16")
    assert_close(c16, o["costs"], rtol=TC_COST_RTOL, atol=1e-3, what="costs")
    for g, n in zip(g16, NAMES):
        assert_close(g, o[n], rtol=0, atol=0, ntol=TC_GRAD_NTOL, what=n)
        rel = np.linalg.norm(g - o[n]) / np.linalg.norm(o[n])
        assert rel < 5e-3, (n, rel)


def test_c3_single_utterance_vs_oracle(oracle):
    """One utterance of the BENCHMARKED configuration (BASELINE C3: T=512 U=128 V=1024 H=640, 65 536 cells, 639-step
    wavefront) against the fp64 oracle: pins the tensor-core path to the oracle at the size whose numerics matter (the
    rounding noise of the log-probs accumulates along the lattice), not only to the repo's own fp32 path."""
    k = synth(1, 512, 128, 1024, 640, 6, ragged=False)
    o = oracle_of(oracle, k, np.ones(1))
    costs, grads = run_joint(k, "bf16", scale=np.ones(1))
    assert_close(costs, o["costs"], rtol=TC_COST_RTOL, atol=0, what="costs")
    for g, n in zip(grads, NAMES):
        rel = np.linalg.norm(g - o[n]) / np.linalg.norm(o[n])
        assert np.all(np.isfinite(g)) and rel < 5e-3, (n, rel)


def test_tc_common_voice_shaped_batch():
    """BASELINE C5 in miniature: ragged T_b, U_b (one long and one minimal utterance), V=4096, H=640, maxU=200 --
    tensor-core path against the fp32 exact path."""
    B, T, U, V, H = 4, 160, 200, 4096, 640
    k = synth(B, T, U, V, H, 11, ragged=False)
    k["input_lengths"] = np.array([T, 10, 97, 160], np.int32)
    k["label_lengths"] = np.array([U - 1, 9, 120, 30], np.int32)
    for b in range(B):
        k["labels"][b, k["label_lengths"][b]:] = 0
    c32, g32 = run_joint(k, "fp32")
    c16, g16 = run_joint(k, "bf16")
    assert np.all(np.isfinite(c16))
    assert_close(c16, c32, rtol=TC_COST_RTOL, atol=1e-3, what="costs")
    for a, b_, n in zip(g16, g32, NAMES):
        assert np.all(np.isfinite(a)), n
        rel = np.linalg.norm(a - b_) / np.linalg.norm(b_)
        assert rel < 5e-3, (n, rel)
    for b in range(B):   # padded positions exactly zero
        assert not g16[0][b, k["input_lengths"][b]:].any() and not g16[1][b, k["label_lengths"][b] + 1:].any()


@pytest.mark.parametrize("B,T,U,V,H,blank", [(3, 9, 1, 64, 64, 0),      # empty transcripts (U == 1)
                                             (3, 1, 5, 64, 128, 0),     # a single encoder frame
                                             (2, 12, 6, 128, 64, 5),    # blank index != 0
                                             (2, 12, 6, 128, 64, 127)]) # blank = last column (last 32-column group)
@pytest.mark.parametrize("keep", [True, False])
def test_tc_edge_lattices(oracle, B, T, U, V, H, blank, keep):
    rng = np.random.default_rng(21)
    k = synth(B, T, max(U, 2), V, H, 21, ragged=False)
    k["pred"] = k["pred"][:, :U].copy()
    cand = np.array([v for v in range(V) if v != blank])
    k["labels"] = rng.choice(cand, size=(B, U - 1)).astype(np.int32) if U > 1 else np.zeros((B, 0), np.int32)
    k["label_lengths"] = np.full(B, U - 1, np.int32)
    k["blank"] = np.int32(blank)
    o = oracle_of(oracle, k, np.full(B, 1.0 / B), blank)
    costs, grads = run_joint(k, "bf16", keep=keep)
    assert_close(costs, o["costs"], rtol=TC_COST_RTOL, atol=1e-3, what="costs")
    for g, n in zip(grads, NAMES):
        assert_close(g, o[n], rtol=0, atol=0, ntol=TC_GRAD_NTOL, what=n)


def test_large_magnitude_logits(oracle):
    """Logits of magnitude ~40 (saturated softmax; the kept bf16 numerators span dozens of binades around the row's
    frame, and a row's maximum lies up to ~28 bits above its first 32 logits -- far below the 2^64 frame switch, which
    tests/test_gpu_joint_extreme_logits.py covers): costs and gradients stay finite and on the oracle."""
    k = synth(2, 24, 10, 128, 64, 9, ragged=True)
    k["W"] = (k["W"] * 12).astype(np.float32)
    k["b"] = (k["b"] * 30).astype(np.float32)
    o = oracle_of(oracle, k, np.full(2, 0.5))
    costs, grads = run_joint(k, "bf16")
    assert np.all(np.isfinite(costs))
    assert_close(costs, o["costs"], rtol=2e-3, atol=1e-2, what="costs")
    for g, n in zip(grads, NAMES):
        assert np.all(np.isfinite(g)), n
        assert_close(g, o[n], rtol=0, atol=0, ntol=2e-2, what=n)


def test_kept_and_recomputed_backward_agree():
    """keep_activations: the backward consumes the numerators the forward call left in the workspace; without it the
    backward re-runs the same keeping forward itself, chunk by chunk.  Same kernels on the same data: identical costs
    (both forward modes use the same arithmetic for the softmax sum) and gradients."""
    k = synth(6, 90, 50, 320, 256, 41, ragged=True)
    c1, g1 = run_joint(k, "bf16", keep=True)
    c2, g2 = run_joint(k, "bf16", keep=False)
    assert np.array_equal(c1, c2)
    for a, b_, n in zip(g1, g2, NAMES):
        assert_close(a, b_, rtol=0, atol=0, ntol=1e-6, what=n)


def test_backward_is_deterministic():
    k = synth(5, 70, 45, 256, 192, 31, ragged=True)
    c1, g1 = run_joint(k, "bf16")
    c2, g2 = run_joint(k, "bf16")
    assert np.array_equal(c1, c2)
    for a, b_, n in zip(g1, g2, NAMES):
        assert np.array_equal(a, b_), n


def test_multi_chunk_backward(tmp_path):
    """Batches whose kept activations exceed one workspace chunk (BASELINE C5) run the backward chunk by chunk.  Forced
    here with RNNTB200_CHUNK_MB=1 (read once per process, hence the child processes): 5 utterances in chunks of 1-2."""
    args = ["5", "70", "45", "256", "192", "31", "1"]
    outs = []
    for tag, env, keep in (("one", {}, "1"), ("chunked", {"RNNTB200_CHUNK_MB": "1"}, "1"), ("chunked_nokeep", {"RNNTB200_CHUNK_MB": "1"}, "0")):
        f = str(tmp_path / (tag + ".npz"))
        subprocess.run([sys.executable, os.path.join(ROOT, "tools", "joint_dump.py"), f] + args + [keep],
                       check=True, env=dict(os.environ, **env), timeout=300)
        outs.append(dict(np.load(f)))
    for o in outs[1:]:
        assert np.array_equal(o["costs"], outs[0]["costs"])
        for n in ("d_enc", "d_pred"):                           # per-utterance quantities
            assert_close(o[n], outs[0][n], rtol=0, atol=0, ntol=1e-6, what=n)
        for n in ("dW", "db"):                                  # summed over utterances in another order
            assert_close(o[n], outs[0][n], rtol=0, atol=0, ntol=2e-5, what=n)


def test_valid_tile_bound_keeps_a_multi_chunk_batch_in_one_chunk(tmp_path):
    """BASELINE C5's situation in miniature: the PADDED numerators of the batch exceed one workspace chunk (forced with
    RNNTB200_CHUNK_MB=1), so by default the backward recomputes chunk by chunk.  With `valid_tiles` (a host-side count of
    the lattice tiles that are actually valid) the workspace holds exactly those row blocks, the batch is ONE chunk and the
    forward keeps its numerators: same costs and gradients, and no recomputing forward launch.  A promise that is too small
    must not write out of bounds: the costs come back NaN."""
    args = ["5", "70", "45", "256", "192", "31", "1", "1"]
    env = dict(os.environ, RNNTB200_CHUNK_MB="1")
    outs = {}
    for tag, bound in (("chunked", "0"), ("bound", "1"), ("broken", "3")):
        f = str(tmp_path / (tag + ".npz"))
        subprocess.run([sys.executable, os.path.join(ROOT, "tools", "joint_dump.py"), f] + args + [bound],
                       check=True, env=env, timeout=300)
        outs[tag] = dict(np.load(f))
    kernels = lambda o: " ".join(str(x) for x in o["kernels"])
    assert "<fwd>" in kernels(outs["chunked"])                      # costs-only forward + recomputing forwards in the backward
    assert "<fwd>" not in kernels(outs["bound"]) and "<fwd+keep>" in kernels(outs["bound"])
    assert np.array_equal(outs["bound"]["costs"], outs["chunked"]["costs"])
    for n in ("d_enc", "d_pred"):
        assert_close(outs["bound"][n], outs["chunked"][n], rtol=0, atol=0, ntol=1e-6, what=n)
    for n in ("dW", "db"):
        assert_close(outs["bound"][n], outs["chunked"][n], rtol=0, atol=0, ntol=2e-5, what=n)
    assert np.isnan(outs["broken"]["costs"]).all()


def test_one_cta_kernel_forms_agree_with_the_pair_kernels(tmp_path):
    """The one-CTA forms of the three tensor-core kernels (RNNTB200_FWD=3, RNNTB200_DZ=1, RNNTB200_DW=1: A/B references of the
    CTA-pair kernels, selected once per process) compute the same function: costs to 1e-5 relative, gradients to the
    16-bit path's own noise level (summation orders differ)."""
    args = ["3", "40", "21", "576", "640", "17", "1", "1"]       # ragged, two dZ passes, two v-tiles (512 + 64), odd u-block counts
    outs = {}
    for tag, env in (("pair", {}), ("one", {"RNNTB200_FWD": "3", "RNNTB200_DZ": "1", "RNNTB200_DW": "1"})):
        f = str(tmp_path / (tag + ".npz"))
        subprocess.run([sys.executable, os.path.join(ROOT, "tools", "joint_dump.py"), f] + args,
                       check=True, env=dict(os.environ, **env), timeout=300)
        outs[tag] = dict(np.load(f))
    k = " ".join(str(x) for x in outs["one"]["kernels"])
    assert "joint_tc3_kernel" in k and "bwd_dw_kernel" in k and "bwd_dw2_kernel" not in k
    assert_close(outs["one"]["costs"], outs["pair"]["costs"], rtol=1e-5, atol=1e-4, what="costs")
    for n in NAMES:
        assert_close(outs["one"][n], outs["pair"][n], rtol=0, atol=0, ntol=2e-3, what=n)


def test_cuda_graph_capture_and_replay():
    """The whole fused forward + backward is stream-ordered (no host synchronisation, no allocation inside the library
    calls): it can be captured into a CUDA graph and replayed on new input values."""
    import rnnt_speech_recognition_b200 as rb
    torch.manual_seed(0)
    B, T, U, V, H = 4, 64, 32, 256, 128
    enc = torch.randn(B, T, H, device="cuda", requires_grad=True)
    pred = torch.randn(B, U, H, device="cuda", requires_grad=True)
    W = (torch.randn(H, V, device="cuda") / H ** 0.5).requires_grad_()
    b = torch.zeros(V, device="cuda", requires_grad=True)
    lab = torch.randint(1, V, (B, U - 1), dtype=torch.int32, device="cuda")
    il = torch.tensor([T, T - 7, 20, T], dtype=torch.int32, device="cuda")
    ll = torch.tensor([U - 1, 5, U - 1, 12], dtype=torch.int32, device="cuda")

    def step():
        for t in (enc, pred, W, b):
            t.grad = None
        costs = rb.joint_rnnt_loss(enc, pred, W, b, lab, il, ll, precision="bf16")
        (costs.sum() / B).backward()
        return costs

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            out = step()
        grads = [t.grad for t in (enc, pred, W, b)]
    torch.cuda.current_stream().wait_stream(s)
    with torch.no_grad():                      # new input values in the captured buffers
        enc.copy_(torch.randn_like(enc))
        pred.copy_(torch.randn_like(pred))
    g.replay()
    torch.cuda.synchronize()
    got_c, got_g = out.clone(), [x.clone() for x in grads]
    want_c = step().detach()
    torch.cuda.synchronize()
    assert torch.equal(got_c, want_c)
    for a, t in zip(got_g, (enc, pred, W, b)):
        assert torch.equal(a, t.grad)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_two_devices_one_process():
    """A MirroredStrategy-style caller (run_rnnt.py:119-127): ONE process drives several GPUs.  The library keeps no
    per-process device state (shared-memory opt-in per device, SM count per call, stream from the descriptor)."""
    k = synth(3, 40, 20, 128, 128, 51, ragged=True)
    import rnnt_speech_recognition_b200 as rb
    res = []
    for dev in (0, 1, 0):
        t = [torch.as_tensor(k[n]).to("cuda:%d" % dev).requires_grad_() for n in ("enc", "pred", "W", "b")]
        ints = [torch.as_tensor(k[n]).to("cuda:%d" % dev) for n in ("labels", "input_lengths", "label_lengths")]
        costs = rb.joint_rnnt_loss(*t, *ints, precision="bf16")
        (costs.sum() / 3).backward()
        res.append((costs.detach().cpu().numpy(), [x.grad.cpu().numpy() for x in t]))
    for c, g in res[1:]:
        assert np.array_equal(c, res[0][0])
        for a, b_ in zip(g, res[0][1]):
            assert np.array_equal(a, b_)
