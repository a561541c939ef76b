#!/usr/bin/env python
"""Generate the committed golden fixtures under tests/golden/ FROM THE REFERENCE.

Run in the build container only (needs /root/reference); the outputs (*.npz) are committed so
that nothing on the GPU box reads /root/reference.

Sources of truth, in order:
  1. The reference's own known-answer tests, parsed (not hand-copied) from
       warp-transducer/pytorch_binding/test/test.py:51-160   (acts, costs, logits-grads)
       warp-transducer/tests/test_cpu.cpp:79-109             (log-prob-grads of the B=2 KAT)
  2. The reference library itself, built unmodified by oracle/Makefile into
       oracle/_ref/libwarprnnt.so and driven through its C ABI (rnnt.h:104-124), on seeded
       random cases covering what the reference tests do not (ragged lengths, U=1, T=1,
       blank != 0, repeated labels, large-magnitude logits).
  3. For the joint network (TensorFlow arithmetic, un-vendored, no pinned vectors in the
       reference): model.py:158-166 restated in torch fp64, chained by autograd through
       torch log_softmax (utils/loss.py:30) into the reference library's fp64 entry point
       (compute_rnnt_loss_fp64, rnnt.h:115-124).
  4. The reference header's ABI (reference_abi.json): the functions rnnt.h declares, the
       rnntOptions layout and enum values that tests/abi_harness reports when it is compiled
       against rnnt.h, and the reference library's version and status strings.
"""
import ast
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import oracle  # noqa: E402

REF = "/root/reference/warp-transducer"


# ------------------------------------------------------------------ 1. parse the reference KATs
def _literal(node):
    """Evaluate a literal / np.array(literal) AST node."""
    if isinstance(node, ast.Call):  # np.array([...])
        return np.array(_literal(node.args[0]))
    return ast.literal_eval(node)


def parse_pytorch_kats():
    src = open(os.path.join(REF, "pytorch_binding/test/test.py")).read()
    tree = ast.parse(src)
    out = {}
    for fn in tree.body:
        if isinstance(fn, ast.FunctionDef) and fn.name in ("small_test", "big_test"):
            vals = {}
            for st in fn.body:
                if isinstance(st, ast.Assign) and isinstance(st.targets[0], ast.Name):
                    name = st.targets[0].id
                    if name in ("acts", "activations", "labels", "expected_cost", "expected_costs",
                                "expected_grads") and name not in vals:
                        vals[name] = _literal(st.value)
            out[fn.name] = vals
    return out


def parse_cpp_vector(path, func, var):
    src = open(path).read()
    body = src[src.index("bool %s()" % func):]
    m = re.search(r"std::vector<\w+>\s+%s\s*=\s*\{([^}]*)\}" % var, body)
    return np.array([float(x) for x in m.group(1).replace("\n", " ").split(",") if x.strip()])


# ------------------------------------------------------------------ 2. reference library drivers
def ref_fp64(log_probs, labels, input_lengths, label_lengths, blank):
    """compute_rnnt_loss_fp64(RNNT_CPU): costs and grads wrt log-probs, double precision."""
    L = oracle.ref()
    lp = np.ascontiguousarray(log_probs, dtype=np.float64)
    B, T, U, V = lp.shape
    labels = np.ascontiguousarray(labels, dtype=np.int32)
    ll = np.ascontiguousarray(label_lengths, dtype=np.int32)
    il = np.ascontiguousarray(input_lengths, dtype=np.int32)
    sz = C.c_size_t(0)
    L.get_workspace_size(T, U, B, False, C.byref(sz), 8)
    ws = np.empty(sz.value, np.uint8)
    costs = np.zeros(B, np.float64)
    grads = np.zeros_like(lp)
    L.compute_rnnt_loss_fp64.argtypes = L.compute_rnnt_loss.argtypes
    rc = L.compute_rnnt_loss_fp64(lp.ctypes.data, grads.ctypes.data, labels.ctypes.data, ll.ctypes.data,
                                  il.ctypes.data, V, B, costs.ctypes.data, ws.ctypes.data,
                                  oracle.RnntOptions(0, 1, None, blank, T, U, True))
    assert rc == 0
    return costs, grads


class RefLoss64(torch.autograd.Function):
    """Reference loss op in fp64 as a torch autograd node (mirrors warprnnt_pytorch _RNNT,
    pytorch_binding/warprnnt_pytorch/__init__.py:10-50: grads cached in forward)."""

    @staticmethod
    def forward(ctx, log_probs, labels, il, ll, blank):
        costs, grads = ref_fp64(log_probs.detach().numpy(), labels, il, ll, blank)
        ctx.grads = torch.from_numpy(grads)
        return torch.from_numpy(costs)

    @staticmethod
    def backward(ctx, go):
        return ctx.grads * go.view(-1, 1, 1, 1), None, None, None, None


def logits_case(rng, B, T, U, V, blank=0, ragged=False, scale=1.0, uniform=False, repeats=False):
    acts = (rng.uniform(0, 1, (B, T, U, V)) if uniform else rng.standard_normal((B, T, U, V)) * scale)
    acts = acts.astype(np.float32)
    cand = [v for v in range(V) if v != blank]
    labels = rng.choice(cand, size=(B, max(U - 1, 1))).astype(np.int32)
    if U == 1:
        labels = np.zeros((B, 0), np.int32)
    if repeats and U >= 4:  # forced repeats, as random.cpp:33-36 does
        L = U - 1
        labels[:, L // 2] = labels[:, L // 2 + 1]
        labels[:, L // 2 - 1] = labels[:, L // 2]
    il = np.full(B, T, np.int32)
    ll = np.full(B, U - 1, np.int32)
    if ragged:
        il = rng.integers(1, T + 1, B).astype(np.int32)
        ll = rng.integers(0, U, B).astype(np.int32)
        il[0], ll[0] = T, U - 1           # certify_inputs: T == max(lengths), U == max(label_lengths)+1
        if B > 1:
            il[1], ll[1] = 1, 0           # smallest lattice in the same batch
        for b in range(B):
            labels[b, ll[b]:] = 0         # zero padding, preprocessing.py padded_batch
    x = torch.tensor(acts, dtype=torch.float64, requires_grad=True)
    costs = RefLoss64.apply(torch.log_softmax(x, -1), labels, il, ll, blank)
    costs.sum().backward()
    # fp32 run of the real reference on fp32 log-probs (what the TF CPU build executes)
    lp32 = torch.log_softmax(torch.tensor(acts), -1).numpy()
    c32, g32 = oracle.ref_cpu_cost_and_grad(lp32, labels, il, ll, blank, num_threads=1)
    return dict(acts=acts, labels=labels, input_lengths=il, label_lengths=ll, blank=np.int32(blank),
                costs=costs.detach().numpy(), logits_grads=x.grad.numpy(), costs_f32=c32, logprob_grads_f32=g32)


def joint_case(rng, B, T, U, V, H, blank=0, ragged=False):
    enc = rng.standard_normal((B, T, H))
    pred = rng.standard_normal((B, U, H))
    W = rng.standard_normal((H, V)) / np.sqrt(H)
    b = rng.standard_normal(V) * 0.1
    # inputs are fp32 values; the fp64 ground truth is computed on exactly those values
    enc, pred, W, b = (a.astype(np.float32).astype(np.float64) for a in (enc, pred, W, b))
    cand = [v for v in range(V) if v != blank]
    labels = rng.choice(cand, size=(B, U - 1)).astype(np.int32)
    il = np.full(B, T, np.int32)
    ll = np.full(B, U - 1, np.int32)
    if ragged:
        il = rng.integers(1, T + 1, B).astype(np.int32)
        ll = rng.integers(0, U, B).astype(np.int32)
        il[0], ll[0] = T, U - 1
        for i in range(B):
            labels[i, ll[i]:] = 0
    t = [torch.tensor(a, dtype=torch.float64, requires_grad=True) for a in (enc, pred, W, b)]
    z = torch.tanh(t[0][:, :, None, :] + t[1][:, None, :, :])      # model.py:158-163
    logits = z @ t[2] + t[3]                                        # model.py:165-166
    costs = RefLoss64.apply(torch.log_softmax(logits, -1), labels, il, ll, blank)  # utils/loss.py:29-35
    (costs.sum() / B).backward()                                    # run_rnnt.py:278
    return dict(enc=enc.astype(np.float32), pred=pred.astype(np.float32), W=W.astype(np.float32),
                b=b.astype(np.float32), labels=labels, input_lengths=il, label_lengths=ll, blank=np.int32(blank),
                costs=costs.detach().numpy(), d_enc=t[0].grad.numpy(), d_pred=t[1].grad.numpy(),
                dW=t[2].grad.numpy(), db=t[3].grad.numpy())


def ref_cpu_case(acts, labels, il, ll, blank):
    """Log-probs of `acts` through the reference's fp32 CPU path: what tests/test_oracle.py holds the oracle to."""
    lp = oracle.log_softmax(acts)
    costs, grads = oracle.ref_cpu_cost_and_grad(lp, labels, il, ll, blank=blank, num_threads=1)
    return dict(log_probs=lp, labels=labels, input_lengths=il, label_lengths=ll, blank=np.int32(blank), costs=costs,
                grads=grads)


def ref_cpu_random_case():
    """Fresh random input, ragged down to a single frame and an empty transcript, plus the reference's GPU workspace size."""
    rng = np.random.default_rng(99)
    B, T, U, V = 4, 13, 6, 9
    acts = rng.standard_normal((B, T, U, V)).astype(np.float32)
    labels = rng.integers(1, V, (B, U - 1)).astype(np.int32)
    k = ref_cpu_case(acts, labels, np.array([13, 7, 1, 10], np.int32), np.array([5, 2, 0, 4], np.int32), 0)
    sz = C.c_size_t(0)
    assert oracle.ref().get_workspace_size(T, U, B, True, C.byref(sz), 4) == 0
    k["gpu_workspace_bytes"] = np.int64(sz.value)
    return k


# (B, T, U, V, seed, logit scale): the 40 examples hypothesis draws (derandomized) from B in [1,4], T in [1,12],
# U in [1,7], V in [2,11], scale in {0.3, 1, 6} -- boundary shapes first, then shrinks of larger ones
PROPERTY_CASES = [
    (1, 1, 1, 2, 0, 0.3), (2, 1, 1, 2, 0, 0.3), (2, 8, 7, 2, 9197, 6.0), (1, 12, 1, 2, 0, 0.3), (1, 12, 6, 5, 104017, 1.0),
    (4, 9, 5, 11, 1764902504, 6.0), (4, 2, 4, 5, 13649451, 1.0), (3, 10, 5, 7, 4466, 1.0), (3, 1, 1, 3, 23782899, 6.0),
    (4, 10, 6, 8, 22369, 6.0), (4, 9, 7, 2, 500, 0.3), (4, 9, 7, 7, 500, 0.3), (4, 9, 1, 7, 500, 0.3), (4, 7, 1, 7, 500, 0.3),
    (4, 7, 1, 4, 500, 0.3), (4, 7, 1, 2, 500, 0.3), (4, 7, 1, 2, 2, 0.3), (4, 1, 2, 10, 532, 6.0), (4, 1, 1, 10, 532, 6.0),
    (4, 1, 1, 2, 532, 6.0), (4, 1, 1, 2, 2, 6.0), (4, 1, 2, 2, 2, 6.0), (4, 2, 2, 2, 2, 6.0), (2, 2, 2, 2, 2, 6.0),
    (2, 9, 3, 2, 99999999, 1.0), (1, 9, 3, 2, 99999999, 1.0), (1, 9, 3, 2, 9, 1.0), (1, 2, 3, 2, 9, 1.0), (1, 2, 1, 2, 9, 1.0),
    (1, 1, 1, 2, 9, 1.0), (1, 1, 1, 2, 1, 1.0), (1, 4, 3, 2, 1561, 6.0), (1, 1, 3, 2, 1561, 6.0), (1, 1, 3, 2, 2, 6.0),
    (1, 1, 3, 2, 1, 6.0), (1, 1, 1, 2, 1, 6.0), (1, 1, 1, 2, 2, 6.0), (4, 8, 1, 6, 3199819, 0.3), (4, 8, 1, 2, 3199819, 0.3),
    (4, 2, 1, 2, 3199819, 0.3)]


def ref_cpu_property_case(B, T, U, V, seed, scale):
    """Random shape, ragged lengths, random blank position and logit scale."""
    rng = np.random.default_rng(seed)
    acts = (scale * rng.standard_normal((B, T, U, V))).astype(np.float32)
    blank = int(rng.integers(0, V))
    cand = np.array([v for v in range(V) if v != blank])
    labels = (rng.choice(cand, size=(B, U - 1)).astype(np.int32) if U > 1 else np.zeros((B, 0), np.int32))
    il = rng.integers(1, T + 1, B).astype(np.int32)
    ll = rng.integers(0, U, B).astype(np.int32)
    il[0], ll[0] = T, U - 1                       # the reference sizes its slabs by maxT / maxU
    return ref_cpu_case(acts, labels, il, ll, blank)


def joint_property_cases():
    """Ten small random joint cases beyond the named fixtures (random blank, half of them ragged)."""
    rng = np.random.default_rng(20260924)
    out = []
    for _ in range(10):
        B, T, U = int(rng.integers(1, 4)), int(rng.integers(1, 9)), int(rng.integers(1, 6))
        V, H = int(rng.integers(2, 9)), int(rng.integers(1, 7))
        out.append(joint_case(rng, B, T, U, V, H, blank=int(rng.integers(0, V)), ragged=bool(rng.integers(0, 2))))
    return out


def save_cases(path, cases):
    """Several cases of different shapes in one .npz: case i's arrays under "c<ii>_<name>"."""
    np.savez_compressed(path, **{"c%02d_%s" % (i, n): a for i, k in enumerate(cases) for n, a in k.items()})


def reference_abi():
    """tests/abi_harness compiled against the reference's rnnt.h (and linked against this library, which it needs to
    link) reports the header's rnntOptions layout and enum values; the version and status strings are the reference
    library's own."""
    hdr = open(os.path.join(REF, "include", "rnnt.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    funcs = sorted(set(re.findall(r"^\s*(?:rnntStatus_t|int|const char\*)\s+(\w+)\s*\(", hdr, flags=re.M)))
    pkg = os.path.join(ROOT, "rnnt_speech_recognition_b200")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "abi_harness")
        subprocess.run(["g++", "-O1", "-std=c++14", "-DRNNT_REFERENCE_HEADER", "-I" + os.path.join(REF, "include"),
                        "-I/usr/local/cuda/include", os.path.join(ROOT, "tests", "abi_harness", "abi_harness.cpp"),
                        "-L" + pkg, "-l:librnnt_b200.so", "-L/usr/local/cuda/lib64", "-lcudart", "-Wl,-rpath," + pkg,
                        "-Wl,-rpath,/usr/local/cuda/lib64", "-o", exe], check=True)
        layout = json.loads(subprocess.run([exe, "layout"], check=True, capture_output=True, text=True).stdout)
    R = oracle.ref()
    return {"header_functions": funcs, "layout": layout, "version": R.get_warprnnt_version(),
            "status_strings": [R.rnntGetStatusString(i).decode() for i in range(6)]}


def main():
    assert oracle.have_ref(), "needs oracle/_ref/libwarprnnt.so (make -C oracle)"
    kats = parse_pytorch_kats()
    s, b = kats["small_test"], kats["big_test"]
    np.savez(os.path.join(HERE, "kat_small.npz"), acts=np.asarray(s["acts"], np.float64),
             labels=np.asarray(s["labels"], np.int32), input_lengths=np.array([2], np.int32),
             label_lengths=np.array([2], np.int32), cost=np.float64(s["expected_cost"]),
             logits_grads=np.asarray(s["expected_grads"], np.float64))
    lp_grads = parse_cpp_vector(os.path.join(REF, "tests/test_cpu.cpp"), "options_test", "expected_grads")
    acts32 = parse_cpp_vector(os.path.join(REF, "tests/test_cpu.cpp"), "options_test", "acts")
    np.savez(os.path.join(HERE, "kat_big.npz"), acts=np.asarray(b["activations"], np.float64),
             acts_6dp=acts32.reshape(2, 4, 3, 3), labels=np.asarray(b["labels"], np.int32),
             input_lengths=np.array([4, 4], np.int32), label_lengths=np.array([2, 2], np.int32),
             costs=np.asarray(b["expected_costs"], np.float64),
             logits_grads=np.asarray(b["expected_grads"], np.float64), logprob_grads=lp_grads.reshape(2, 4, 3, 3))

    rng = np.random.default_rng(1234)
    cases = {
        "inf_shape_T50_U10_V15": logits_case(rng, 1, 50, 10, 15, uniform=True, repeats=True),
        "gradcheck_V20_T50_U15_B1": logits_case(rng, 1, 50, 15, 20, uniform=True, repeats=True),
        "gradcheck_V5_T10_U5_B65": logits_case(rng, 65, 10, 5, 5, uniform=True, repeats=True),
        "ragged_B5_T12_U7_V11": logits_case(rng, 5, 12, 7, 11, ragged=True),
        "u1_empty_transcript": logits_case(rng, 3, 9, 1, 6),
        "t1_single_frame": logits_case(rng, 3, 1, 5, 6),
        "blank3": logits_case(rng, 2, 8, 6, 7, blank=3, ragged=True),
        "large_magnitude": logits_case(rng, 2, 10, 6, 9, scale=30.0),
        "wide_U70_V40": logits_case(rng, 2, 24, 70, 40, ragged=True),
    }
    for k, v in cases.items():
        np.savez_compressed(os.path.join(HERE, "logits_%s.npz" % k), **v)
    jc = {
        "c1_B2_T20_U8_V32_H64": joint_case(rng, 2, 20, 8, 32, 64),
        "ragged_B3_T9_U6_V16_H24": joint_case(rng, 3, 9, 6, 16, 24, ragged=True),
        "blank2_B2_T7_U5_V12_H40": joint_case(rng, 2, 7, 5, 12, 40, blank=2),
    }
    for k, v in jc.items():
        np.savez_compressed(os.path.join(HERE, "joint_%s.npz" % k), **v)
    np.savez_compressed(os.path.join(HERE, "refcpu_random_B4_T13_U6_V9.npz"), **ref_cpu_random_case())
    save_cases(os.path.join(HERE, "refcpu_property_cases.npz"), [ref_cpu_property_case(*c) for c in PROPERTY_CASES])
    save_cases(os.path.join(HERE, "jointchain_property_cases.npz"), joint_property_cases())
    with open(os.path.join(HERE, "reference_abi.json"), "w") as f:
        json.dump(reference_abi(), f, indent=1)
        f.write("\n")
    print("wrote", len(cases) + len(jc) + 6, "fixtures to", HERE)


if __name__ == "__main__":
    main()
