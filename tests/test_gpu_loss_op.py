"""GPU parity of the loss op on materialised logits, THROUGH THE C ABI (compute_rnnt_loss et al.),
against the reference's known-answer tests, the golden fixtures and the CPU oracle."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import assert_close, fp32_tol, golden_names, load

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def L():
    from rnnt_speech_recognition_b200 import _lib
    return _lib.load()


def dev(a, dtype=None):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).cuda()


def c_abi_loss(L, acts, labels, il, ll, blank=0, want_grad=True, fp64=False):
    """compute_rnnt_loss exactly as the reference's bindings call it (warprnnt_op.cc:105-141):
    device acts/labels/lengths/workspace, HOST costs."""
    from rnnt_speech_recognition_b200 import _lib
    dt = torch.float64 if fp64 else torch.float32
    x = dev(acts, dt)
    B, T, U, V = x.shape
    lab = dev(labels, torch.int32) if np.size(labels) else torch.zeros(1, dtype=torch.int32).cuda()
    d_il, d_ll = dev(il, torch.int32), dev(ll, torch.int32)
    sz = C.c_size_t(0)
    assert L.get_workspace_size(T, U, B, True, C.byref(sz), 8 if fp64 else 4) == 0
    ws = torch.empty(sz.value, dtype=torch.uint8, device="cuda")
    g = torch.full_like(x, float("nan")) if want_grad else None
    costs = np.zeros(B, np.float64 if fp64 else np.float32)
    opt = _lib.RnntOptions(_lib.RNNT_GPU, 0, torch.cuda.current_stream().cuda_stream, blank, T, U, True)
    fn = L.compute_rnnt_loss_fp64 if fp64 else L.compute_rnnt_loss
    st = fn(x.data_ptr(), g.data_ptr() if want_grad else None, lab.data_ptr(), d_ll.data_ptr(), d_il.data_ptr(), V, B,
            costs.ctypes.data, ws.data_ptr(), opt)
    assert st == 0, L.rnntGetStatusString(st)
    return costs, (g.cpu().numpy() if want_grad else None)


def test_kat_small(L):
    k = load("kat_small.npz")      # tests/test_gpu.cu:18-94, pytorch_binding/test/test.py:51-78
    costs, g = c_abi_loss(L, k["acts"], k["labels"], k["input_lengths"], k["label_lengths"])
    assert abs(costs[0] - k["cost"]) < 1e-4
    assert np.allclose(g, k["logits_grads"], atol=1e-6)
    c2, _ = c_abi_loss(L, k["acts"], k["labels"], k["input_lengths"], k["label_lengths"], want_grad=False)
    assert np.allclose(c2, costs)  # score_forward (gradients == NULL)


def test_kat_big(L):
    k = load("kat_big.npz")        # tests/test_gpu.cu:96-224, test_warprnnt_op.py:52-87
    costs, g = c_abi_loss(L, k["acts"], k["labels"], k["input_lengths"], k["label_lengths"])
    assert np.allclose(costs, k["costs"], atol=1e-6, rtol=1e-6)
    assert np.allclose(g, k["logits_grads"], atol=1e-6)          # atol of test_warprnnt_op.py:25-26
    c64, g64 = c_abi_loss(L, k["acts"], k["labels"], k["input_lengths"], k["label_lengths"], fp64=True)
    assert np.allclose(c64, k["costs"], atol=1e-12) and np.allclose(g64, k["logits_grads"], atol=2e-7)


@pytest.mark.parametrize("name", golden_names("logits_"))
def test_golden_logits_cases(L, name):
    k = load(name)
    blank = int(k["blank"])
    costs, g = c_abi_loss(L, k["acts"], k["labels"], k["input_lengths"], k["label_lengths"], blank)
    assert np.all(np.isfinite(costs)) and np.all(np.isfinite(g))                 # inf_test
    tol = fp32_tol(k["costs"])
    assert_close(costs, k["costs"], rtol=1e-5, atol=1e-5, what="costs")
    assert_close(g, k["logits_grads"], what="logits grads", **tol)
    for b in range(g.shape[0]):                                                  # padded cells exactly 0
        T, U = int(k["input_lengths"][b]), int(k["label_lengths"][b]) + 1
        assert not g[b, T:].any() and not g[b, :, U:].any()
    c64, g64 = c_abi_loss(L, k["acts"], k["labels"], k["input_lengths"], k["label_lengths"], blank, fp64=True)
    assert np.allclose(c64, k["costs"], rtol=1e-10) and np.allclose(g64, k["logits_grads"], atol=1e-10)


@pytest.mark.parametrize("B,T,U,V,seed", [(3, 40, 33, 50, 0), (2, 70, 130, 24, 1), (4, 300, 20, 128, 2),
                                           (1, 5, 257, 10, 3)])
def test_random_vs_oracle(L, oracle, B, T, U, V, seed):
    """Multi-warp wavefronts (U > 32), ragged lengths, vocab not a multiple of 32."""
    rng = np.random.default_rng(seed)
    acts = rng.standard_normal((B, T, U, V)).astype(np.float32)
    labels = rng.integers(1, V, (B, U - 1)).astype(np.int32)
    il = rng.integers(1, T + 1, B).astype(np.int32)
    ll = rng.integers(0, U, B).astype(np.int32)
    il[0], ll[0] = T, U - 1
    oc, og = oracle.rnnt_logits_grad(acts.astype(np.float64), labels, il, ll)
    costs, g = c_abi_loss(L, acts, labels, il, ll)
    assert_close(costs, oc, rtol=1e-5, atol=1e-4, what="costs")
    assert_close(g, og, what="grads", **fp32_tol(oc))


def test_torch_surface_matches_reference_bindings():
    """rnnt_loss (TF signature), torch_rnnt_loss reductions, RNNTLoss, get_loss_fn."""
    import rnnt_speech_recognition_b200 as rb
    k = load("kat_big.npz")
    x = dev(k["acts"], torch.float32).requires_grad_()
    lab, il, ll = dev(k["labels"], torch.int32), dev(k["input_lengths"], torch.int32), dev(k["label_lengths"], torch.int32)
    costs = rb.rnnt_loss(x, lab, il, ll)
    assert costs.is_cuda and costs.shape == (2,)
    assert np.allclose(costs.detach().cpu().numpy(), k["costs"], atol=1e-6)
    costs.sum().backward()
    assert np.allclose(x.grad.cpu().numpy(), k["logits_grads"], atol=1e-6)
    # _RNNTLossGrad: upstream gradient broadcast per utterance (warprnnt_tensorflow/__init__.py:37-42)
    x2 = dev(k["acts"], torch.float32).requires_grad_()
    (rb.rnnt_loss(x2, lab, il, ll) * torch.tensor([2.0, -0.5]).cuda()).sum().backward()
    want = k["logits_grads"] * np.array([2.0, -0.5])[:, None, None, None]
    assert np.allclose(x2.grad.cpu().numpy(), want, atol=2e-6)
    # warprnnt_pytorch reductions (warprnnt_pytorch/__init__.py:36-40)
    for red, scale in (("sum", 1.0), ("mean", 0.5)):
        x3 = dev(k["acts"], torch.float32).requires_grad_()
        out = rb.RNNTLoss(reduction=red)(x3, lab, il, ll)
        assert out.shape == (1,) and abs(out.item() - k["costs"].sum() * scale) < 1e-5
        out.backward()
        assert np.allclose(x3.grad.cpu().numpy(), k["logits_grads"] * scale, atol=1e-6)
    # utils/loss.get_loss_fn: spec lengths are pre-reduction frame counts (ceil(7/2) == ceil(8/2) == 4)
    loss_fn = rb.get_loss_fn(2)
    c = loss_fn(lab.long(), x.detach(), torch.tensor([7, 8]).cuda(), ll.long())
    assert np.allclose(c.cpu().numpy(), k["costs"], atol=1e-6)


def test_forward_backward_likelihood_agree(L):
    """cost_and_grad_kernel's sanity check (cpu_rnnt.h:166-170): llForward == llBackward, here at the
    BASELINE C2 lattice size and through the device-cost entry."""
    import rnnt_speech_recognition_b200 as rb
    torch.manual_seed(0)
    B, T, U, V = 4, 256, 64, 64
    x = torch.randn(B, T, U, V, device="cuda", requires_grad=True)
    lab = torch.randint(1, V, (B, U - 1), dtype=torch.int32, device="cuda")
    il = torch.full((B,), T, dtype=torch.int32, device="cuda")
    ll = torch.full((B,), U - 1, dtype=torch.int32, device="cuda")
    costs = rb.rnnt_loss(x, lab, il, ll)
    costs.sum().backward()
    g = x.grad
    # every cell's gradient row sums to zero: exp(alpha+beta-ll) splits exactly into its two outgoing arcs
    # (to fp32 round-off of exponents of magnitude |cost| ~ 1.5e3: a few 1e-4)
    assert g.sum(-1).abs().max().item() < 2e-3
    # independent check of the costs: torch log_softmax + the same lattice evaluated per utterance on CPU (fp64)
    from oracle import oracle as o
    oc, _ = o.rnnt_logits_grad(x.detach().cpu().double().numpy(), lab.cpu().numpy(), il.cpu().numpy(),
                               ll.cpu().numpy(), want_grad=False)
    assert_close(costs.detach().cpu().numpy(), oc, rtol=2e-6, atol=1e-3, what="C2-lattice costs")


def test_abi_harness_kat():
    """The C++ harness that uses the warp-transducer API through include/rnnt_b200.h (tests/abi_harness) runs the
    reference's small_test KAT (tests/test_cpu.cpp:12-71) through compute_rnnt_loss on the GPU: cost 4.495666 and the
    first gradient row."""
    import subprocess
    import __graft_entry__ as ge
    exe = ge.build_abi_harness()
    r = subprocess.run([exe, "run"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "run ok" in r.stdout
