"""The tensor-core path at any vocabulary size V >= 1 and any joint width 1 <= H <= 768.  The kernels run the padded problem
(ceil64(H), ceil64(V)) whose padding contributes exactly zero: checked against the fp64 oracle, against the recorded golden
fixtures, bit for bit against the explicitly padded aligned problem, and against the fp32 path at realistic batch sizes."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, assert_close, golden_names, load
from test_gpu_joint import run_joint, synth
from test_gpu_joint_bf16 import NAMES, TC_COST_RTOL, TC_GRAD_NTOL, oracle_of

pytestmark = pytest.mark.gpu


def with_blank(k, blank, seed):
    """Labels drawn from every class but `blank`."""
    B, U1 = k["labels"].shape
    V = k["W"].shape[1]
    rng = np.random.default_rng(seed)
    cand = np.array([v for v in range(V) if v != blank])
    k["labels"] = rng.choice(cand, size=(B, U1)).astype(np.int32)
    k["blank"] = np.int32(blank)
    return k


@pytest.mark.parametrize("B,T,U,V,H,blank,seed", [
    (3, 37, 19, 31, 640, 0, 0),       # character vocabulary of the reference, ragged
    (2, 20, 9, 2, 64, 0, 1),          # smallest useful vocabulary
    (3, 25, 11, 33, 50, 32, 2),       # the reference's small joint; blank = 32 sits in the partial column group
    (2, 18, 7, 100, 1, 0, 3),         # H = 1
    (2, 24, 10, 1000, 600, 0, 4),     # Hp = 640: two dZ passes
    (2, 20, 9, 1025, 640, 0, 5),      # the last 64-column chunk holds one real column
    (2, 17, 9, 4095, 256, 0, 6),      # bias table in shared memory
    (2, 16, 8, 4097, 128, 0, 7),      # Vp = 4160: bias read from global memory
    (2, 19, 9, 130, 767, 0, 8),       # Hp = 768
])
@pytest.mark.parametrize("keep", [True, False])
def test_any_size_vs_oracle(oracle, B, T, U, V, H, blank, seed, keep):
    k = with_blank(synth(B, T, U, V, H, seed, ragged=True), blank, seed)
    gs = np.linspace(0.5, 1.5, B)
    o = oracle_of(oracle, k, gs, blank)
    costs, grads = run_joint(k, "bf16", scale=gs, keep=keep)
    assert_close(costs, o["costs"], rtol=TC_COST_RTOL, atol=1e-3, what="costs")
    for g, n in zip(grads, NAMES):
        assert g.shape == o[n].shape, n
        assert_close(g, o[n], rtol=0, atol=0, ntol=TC_GRAD_NTOL, what=n)
    for b in range(B):       # padded positions of d_enc / d_pred are exactly zero
        assert not grads[0][b, k["input_lengths"][b]:].any()
        assert not grads[1][b, k["label_lengths"][b] + 1:].any()


@pytest.mark.parametrize("name", golden_names("joint_"))
def test_golden_joint_bf16(name):
    """The recorded fp64-chain fixtures (V = 32 / 16 / 12, H = 64 / 24 / 40, one with blank = 2) on the tensor cores."""
    k = load(name)
    costs, grads = run_joint(k, "bf16")
    assert_close(costs, k["costs"], rtol=TC_COST_RTOL, atol=1e-3, what="costs")
    for g, n in zip(grads, NAMES):
        assert_close(g, k[n], rtol=0, atol=0, ntol=TC_GRAD_NTOL, what=n)


def pad_problem(k, Hp, Vp):
    """The aligned problem the library runs internally: zero enc / pred / W padding, bias padding -1e30."""
    B, T, H = k["enc"].shape
    U, V = k["pred"].shape[1], k["W"].shape[1]
    q = dict(k)
    q["enc"] = np.zeros((B, T, Hp), np.float32)
    q["enc"][:, :, :H] = k["enc"]
    q["pred"] = np.zeros((B, U, Hp), np.float32)
    q["pred"][:, :, :H] = k["pred"]
    q["W"] = np.zeros((Hp, Vp), np.float32)
    q["W"][:H, :V] = k["W"]
    q["b"] = np.full(Vp, -1e30, np.float32)
    q["b"][:V] = k["b"]
    return q


@pytest.mark.parametrize("B,T,U,V,H,seed", [(3, 37, 19, 31, 50, 0), (2, 24, 10, 1000, 600, 1), (2, 16, 8, 4097, 128, 2),
                                            (2, 20, 9, 130, 640, 3)])
@pytest.mark.parametrize("keep", [True, False])
def test_padding_is_exactly_the_padded_problem(B, T, U, V, H, seed, keep):
    """Same kernels on the same data: an unaligned call and the aligned call on its explicitly padded twin agree bit for bit."""
    k = synth(B, T, U, V, H, seed, ragged=True)
    q = pad_problem(k, (H + 63) // 64 * 64, (V + 63) // 64 * 64)
    c1, g1 = run_joint(k, "bf16", keep=keep)
    c2, g2 = run_joint(q, "bf16", keep=keep)
    assert np.array_equal(c1, c2)
    want = (g2[0][:, :, :H], g2[1][:, :, :H], g2[2][:H, :V], g2[3][:V])
    for a, b_, n in zip(g1, want, NAMES):
        assert a.shape == b_.shape and np.array_equal(a, b_), n


@pytest.mark.parametrize("B,T,U,V,H,seed", [(8, 256, 96, 31, 640, 12), (4, 200, 64, 4073, 640, 13)])
def test_realistic_batches_vs_fp32(B, T, U, V, H, seed):
    """The reference's character and word-piece vocabularies at training batch sizes, against the fp32 CUDA-core path."""
    k = synth(B, T, U, V, H, seed, ragged=True)
    c32, g32 = run_joint(k, "fp32")
    c16, g16 = run_joint(k, "bf16")
    assert np.all(np.isfinite(c16))
    assert_close(c16, c32, rtol=TC_COST_RTOL, atol=1e-3, what="costs")
    for a, b_, n in zip(g16, g32, NAMES):
        assert np.all(np.isfinite(a)), n
        rel = np.linalg.norm(a - b_) / np.linalg.norm(b_)
        assert rel < 5e-3, (n, rel)


def dump(tmp_path, tag, args, env):
    f = str(tmp_path / (tag + ".npz"))
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "joint_dump.py"), f] + args,
                   check=True, env=dict(os.environ, **env), timeout=300)
    return dict(np.load(f))


def test_one_cta_kernel_forms_at_an_unaligned_shape(tmp_path):
    """RNNTB200_FWD=3 / DZ=1 / DW=1 (the one-CTA kernels) compute what the pair kernels compute at V = 1000, H = 600."""
    args = ["3", "40", "21", "1000", "600", "17", "1", "1"]
    pair = dump(tmp_path, "pair", args, {})
    one = dump(tmp_path, "one", args, {"RNNTB200_FWD": "3", "RNNTB200_DZ": "1", "RNNTB200_DW": "1"})
    ks = " ".join(str(x) for x in one["kernels"])
    assert "joint_tc3_kernel" in ks and "bwd_dw_kernel" in ks and "bwd_dw2_kernel" not in ks
    assert_close(one["costs"], pair["costs"], rtol=1e-5, atol=1e-4, what="costs")
    for n in NAMES:
        assert_close(one[n], pair[n], rtol=0, atol=0, ntol=2e-3, what=n)


def test_multi_chunk_backward_at_an_unaligned_shape(tmp_path):
    """RNNTB200_CHUNK_MB=1 forces one utterance chunk per utterance at V = 1000, H = 600, in both keep modes."""
    args = ["5", "70", "45", "1000", "600", "31", "1"]
    one = dump(tmp_path, "one", args + ["1"], {})
    for keep in ("1", "0"):
        o = dump(tmp_path, "chunked" + keep, args + [keep], {"RNNTB200_CHUNK_MB": "1"})
        assert np.array_equal(o["costs"], one["costs"])
        for n in ("d_enc", "d_pred"):
            assert_close(o[n], one[n], rtol=0, atol=0, ntol=1e-6, what=n)
        for n in ("dW", "db"):
            assert_close(o[n], one[n], rtol=0, atol=0, ntol=2e-5, what=n)


def test_cuda_graph_capture_and_replay_unaligned():
    """The staging and narrowing launches of an unaligned H are stream-ordered like the rest: capture and replay."""
    import rnnt_speech_recognition_b200 as rb
    torch.manual_seed(0)
    B, T, U, V, H = 4, 64, 32, 31, 50
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
    with torch.no_grad():
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


def test_joint_module_with_the_reference_vocabulary():
    """rb.Joint(P, 640, 31) at its default precision trains; its gradients agree with the same module on the fp32 path."""
    import rnnt_speech_recognition_b200 as rb
    torch.manual_seed(5)
    B, T, U, P, H, V = 4, 60, 20, 320, 640, 31
    j16 = rb.Joint(P, H, V).cuda()
    j32 = rb.Joint(P, H, V, precision="fp32").cuda()
    j32.load_state_dict(j16.state_dict())
    f, g = torch.randn(B, T, P, device="cuda"), torch.randn(B, U, P, device="cuda")
    lab = torch.randint(1, V, (B, U - 1), dtype=torch.int32, device="cuda")
    il = torch.tensor([T, 41, 17, T], dtype=torch.int32, device="cuda")
    ll = torch.tensor([U - 1, 12, 3, U - 1], dtype=torch.int32, device="cuda")
    grads = []
    for j in (j16, j32):
        fi, gi = f.clone().requires_grad_(), g.clone().requires_grad_()
        costs = j.loss(fi, gi, lab, il, ll)
        costs.sum().backward()
        grads.append([p.grad for p in j.parameters()] + [fi.grad, gi.grad])
    for a, b_ in zip(*grads):
        assert torch.isfinite(a).all()
        rel = float(torch.linalg.norm(a - b_) / torch.linalg.norm(b_))
        assert rel < 5e-3, rel
    # and a training step through joint_train_step on the tensor-core path
    opt = rb.make_optimizer(j16.parameters(), learning_rate=0.02)
    spec = 2 * il
    losses = [rb.joint_train_step(j16, opt, f, g, lab, spec, ll, global_batch_size=B).item() for _ in range(4)]
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses


def test_width_above_768_is_refused_on_the_tensor_cores(capfd):
    k = synth(2, 8, 4, 31, 769, 9, ragged=False)
    with pytest.raises(RuntimeError, match="invalid value"):
        run_joint(k, "bf16")
    assert "768" in capfd.readouterr().err
    costs, grads = run_joint(k, "fp32")
    assert np.all(np.isfinite(costs)) and all(np.all(np.isfinite(g)) for g in grads)
