"""Pin the oracle (oracle/rnnt_oracle.c) against the reference's own known-answer tests and the
golden fixtures generated from the unmodified reference library (tests/golden/make_golden.py)."""
import numpy as np
import pytest

from conftest import assert_close, fp32_tol, golden_names, load


def load_cases(name):
    """The cases of a multi-case fixture (tests/golden/make_golden.py: save_cases), in order."""
    k = load(name)
    n = len({key.split("_", 1)[0] for key in k})
    return [{key.split("_", 1)[1]: v for key, v in k.items() if key.startswith("c%02d_" % i)} for i in range(n)]


def softmax_chain(lp_grads, log_probs):
    """grads wrt logits from grads wrt log-probs: g - P * sum_v g (autograd of log_softmax)."""
    P = np.exp(log_probs.astype(np.float64))
    return lp_grads - P * lp_grads.sum(-1, keepdims=True)


def test_kat_small(oracle):
    k = load("kat_small.npz")   # warp-transducer/tests/test_cpu.cpp:12-71, pytorch test.py:51-78
    acts = k["acts"].astype(np.float32)
    lp = oracle.log_softmax(acts)
    costs, _ = oracle.rnnt_cost_and_grad(lp, k["labels"], k["input_lengths"], k["label_lengths"], want_grad=False)
    assert abs(costs[0] - k["cost"]) < 1e-4            # eps of test_cpu.cpp:66
    c2, g = oracle.rnnt_logits_grad(acts, k["labels"], k["input_lengths"], k["label_lengths"])
    assert np.allclose(c2, k["cost"], rtol=1e-6)       # test.py:75
    assert np.allclose(g, k["logits_grads"])           # test.py:77 (default rtol 1e-5, atol 1e-8)


def test_kat_big_logprob_grads(oracle):
    k = load("kat_big.npz")     # options_test, test_cpu.cpp:73-179
    lp = oracle.log_softmax(k["acts_6dp"].astype(np.float32))
    costs, grads = oracle.rnnt_cost_and_grad(lp, k["labels"], k["input_lengths"], k["label_lengths"])
    assert np.all(np.abs(costs - k["costs"]) < 1e-4)
    assert np.all(np.abs(grads - k["logprob_grads"]) < 1e-4)


def test_kat_big_logits_grads(oracle):
    k = load("kat_big.npz")     # test_gpu.cu:96-224, test_warprnnt_op.py:52-87, test.py:80-160
    costs, grads = oracle.rnnt_logits_grad(k["acts"].astype(np.float32), k["labels"], k["input_lengths"],
                                           k["label_lengths"])
    assert np.allclose(costs, k["costs"], atol=1e-6, rtol=1e-6)
    assert np.allclose(grads, k["logits_grads"], atol=1e-6, rtol=1e-3)
    c64, g64 = oracle.rnnt_logits_grad(k["acts"], k["labels"], k["input_lengths"], k["label_lengths"])
    assert np.allclose(c64, k["costs"], atol=1e-12, rtol=1e-12)
    assert np.allclose(g64, k["logits_grads"], atol=2e-7)   # the KAT table itself was printed from an fp32 run


@pytest.mark.parametrize("name", golden_names("logits_"))
def test_logits_cases(oracle, name):
    k = load(name)
    blank = int(k["blank"])
    costs, grads = oracle.rnnt_logits_grad(k["acts"], k["labels"], k["input_lengths"], k["label_lengths"], blank)
    assert np.all(np.isfinite(costs)) and np.all(np.isfinite(grads))      # inf_test, test_cpu.cpp:181-240
    tol = fp32_tol(k["costs"])
    assert np.allclose(costs, k["costs"], rtol=1e-5, atol=1e-5)
    assert np.allclose(grads, k["logits_grads"], **tol)
    # CPU-path semantics against the fp32 run of the real reference
    lp = oracle.log_softmax(k["acts"])
    c32, g32 = oracle.rnnt_cost_and_grad(lp, k["labels"], k["input_lengths"], k["label_lengths"], blank)
    assert np.allclose(c32, k["costs_f32"], rtol=1e-5, atol=1e-5)
    assert np.allclose(g32, k["logprob_grads_f32"], **tol)
    # padded cells carry exactly zero gradient (gpu_rnnt.h:109, cpu_rnnt.h:155-158)
    for b in range(k["acts"].shape[0]):
        T, U = int(k["input_lengths"][b]), int(k["label_lengths"][b]) + 1
        assert not grads[b, T:].any() and not grads[b, :, U:].any()
    # f64 instantiation agrees with the f64 reference run to round-off
    c64, g64 = oracle.rnnt_logits_grad(k["acts"].astype(np.float64), k["labels"], k["input_lengths"],
                                       k["label_lengths"], blank)
    assert np.allclose(c64, k["costs"], rtol=1e-10) and np.allclose(g64, k["logits_grads"], atol=1e-10)


@pytest.mark.parametrize("name", golden_names("joint_"))
def test_joint_cases(oracle, name):
    k = load(name)
    B = k["enc"].shape[0]
    out = oracle.joint_loss_grad(k["enc"], k["pred"], k["W"], k["b"], k["labels"], k["input_lengths"],
                                 k["label_lengths"], int(k["blank"]), grad_scale=np.full(B, 1.0 / B))
    assert np.allclose(out["costs"], k["costs"], rtol=1e-5)
    for g in ("d_enc", "d_pred", "dW", "db"):
        assert_close(out[g], k[g], rtol=1e-4, atol=1e-6, ntol=1e-5, what=g)
    o64 = oracle.joint_loss_grad(*(k[n].astype(np.float64) for n in ("enc", "pred", "W", "b")), k["labels"],
                                 k["input_lengths"], k["label_lengths"], int(k["blank"]),
                                 grad_scale=np.full(B, 1.0 / B))
    for g in ("d_enc", "d_pred", "dW", "db"):
        assert np.allclose(o64[g], k[g], rtol=1e-9, atol=1e-11), g


def test_numeric_gradient(oracle):
    """Central-difference check, the property test of test_cpu.cpp:287-379 (eps 1e-2, rel-L2 < 1e-4),
    run in fp64 so the finite difference itself is trustworthy."""
    rng = np.random.default_rng(7)
    B, T, U, V = 2, 6, 4, 5
    acts = rng.uniform(0, 1, (B, T, U, V))
    labels = rng.integers(1, V, (B, U - 1)).astype(np.int32)
    il, ll = np.array([T, T - 2], np.int32), np.array([U - 1, U - 2], np.int32)
    _, g = oracle.rnnt_logits_grad(acts, labels, il, ll)
    num = np.zeros_like(acts)
    eps = 1e-4
    flat = acts.reshape(-1)
    for i in range(flat.size):
        old = flat[i]
        flat[i] = old + eps
        cp, _ = oracle.rnnt_logits_grad(acts, labels, il, ll, want_grad=False)
        flat[i] = old - eps
        cm, _ = oracle.rnnt_logits_grad(acts, labels, il, ll, want_grad=False)
        flat[i] = old
        num.reshape(-1)[i] = (cp.sum() - cm.sum()) / (2 * eps)
    rel = ((g - num) ** 2).sum() / (g ** 2).sum()     # rel_diff, tests/test.h:22-32
    assert rel < 1e-8


def test_against_live_reference(oracle):
    """The restatement agrees with the unmodified reference library's fp32 CPU path (its costs and log-prob gradients,
    recorded in tests/golden/refcpu_random_B4_T13_U6_V9.npz) on random input ragged down to a single frame and an
    empty transcript, and sizes the GPU workspace as the reference does."""
    k = load("refcpu_random_B4_T13_U6_V9.npz")
    lp = k["log_probs"]
    B, T, U, V = lp.shape
    c, g = oracle.rnnt_cost_and_grad(lp, k["labels"], k["input_lengths"], k["label_lengths"], int(k["blank"]))
    assert np.allclose(c, k["costs"], rtol=1e-6) and np.allclose(g, k["grads"], rtol=1e-5, atol=1e-7)
    assert oracle.get_workspace_size(T, U, B, True) == (0, int(k["gpu_workspace_bytes"]))


def test_invalid_arguments(oracle):
    assert oracle.get_workspace_size(0, 3, 2, False)[0] == 2    # rnnt_entrypoint.cpp:102-105
    assert oracle.get_workspace_size(4, 3, 2, False) == (0, 2 * 4 * 4 * 3 * 4)
    assert oracle.get_workspace_size(4, 3, 2, True) == (0, 2 * (3 * 4 * 3 + 2) * 4)


def test_against_live_reference_property(oracle):
    """Property-based pin: on the 40 random shapes, ragged lengths, blank positions and logit scales that hypothesis drew
    (tests/golden/make_golden.py: PROPERTY_CASES) the restatement and the unmodified reference library agree on costs
    and log-prob gradients."""
    cases = load_cases("refcpu_property_cases.npz")
    assert len(cases) == 40
    for k in cases:
        lp, blank = k["log_probs"], int(k["blank"])
        c, g = oracle.rnnt_cost_and_grad(lp, k["labels"], k["input_lengths"], k["label_lengths"], blank=blank)
        assert np.allclose(c, k["costs"], rtol=1e-5, atol=1e-6), (lp.shape, blank)
        assert np.allclose(g, k["grads"], rtol=1e-4, atol=1e-6), (lp.shape, blank)


def test_joint_oracle_against_torch_fp64_chain_property(oracle):
    """The joint is parity-unpinned by the reference (TensorFlow arithmetic): its anchor is model.py:158-166 restated in
    torch fp64 and chained by autograd through log_softmax into the reference library's fp64 entry point
    (tests/golden/make_golden.py: joint_case).  Ten random shapes here, beyond the named joint fixtures."""
    cases = load_cases("jointchain_property_cases.npz")
    assert len(cases) == 10
    for k in cases:
        B, T, H = k["enc"].shape
        U, V = k["pred"].shape[1], k["W"].shape[1]
        o64 = oracle.joint_loss_grad(*(k[n].astype(np.float64) for n in ("enc", "pred", "W", "b")), k["labels"],
                                     k["input_lengths"], k["label_lengths"], int(k["blank"]), grad_scale=np.full(B, 1.0 / B))
        assert np.allclose(o64["costs"], k["costs"], rtol=1e-10), (B, T, U, V, H)
        for g in ("d_enc", "d_pred", "dW", "db"):
            assert np.allclose(o64[g], k[g], rtol=1e-9, atol=1e-11), (g, B, T, U, V, H)
