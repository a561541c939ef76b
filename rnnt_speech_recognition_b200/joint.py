"""Fused joint network + RNN-T loss (the north-star path): torch surface over
``rnntb200_joint_loss_forward/backward`` (include/rnnt_b200.h).

Reference being replaced (file:line under /root/reference):
  model.py:158-166      joint_inp = enc[:,:,None,:] + pred[:,None,:,:]; Dense(tanh); Dense(vocab)
  utils/loss.py:24-36   loss adapter -> warprnnt_tensorflow.rnnt_loss
  run_rnnt.py:269-284   model(...) -> loss_fn(...) -> tape.gradient

``enc_acts`` / ``pred_acts`` are the Dense-1 projections hoisted out of the lattice
(W1^T(f_t+g_u)+b1 = (W1^T f_t + b1) + W1^T g_u, SURVEY 8a2): the (B,T,U,*) tensors of the
reference never exist here, in either direction.
"""
import ctypes as C
import os

import torch

from . import _lib
from .loss import encoder_lengths

__all__ = ["joint_rnnt_loss", "joint_logits", "joint_step", "Joint", "get_fused_loss_fn"]

_PREC = {"fp32": _lib.FP32_EXACT, "bf16": _lib.BF16_TC, _lib.FP32_EXACT: _lib.FP32_EXACT, _lib.BF16_TC: _lib.BF16_TC}


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def valid_tile_count(input_lengths, label_lengths):
    """Number of 16 x 8 lattice tiles that intersect the valid lattices of a batch, from HOST copies of the lengths (lists,
    numpy arrays or CPU tensors): the value `joint_rnnt_loss(..., valid_tiles=...)` / `rnntb200JointDesc.valid_tile_bound`
    expects.  A data loader has the lengths on the host anyway; the library itself never reads device memory back."""
    return int(sum(((int(t) + 15) // 16) * ((int(u) + 1 + 7) // 8) for t, u in zip(input_lengths, label_lengths)))


def _desc(B, T, U, H, V, blank, precision, keep=False, tile_bound=0):
    # (call inside `with torch.cuda.device(...)`: the stream is the CURRENT stream of the tensors' device)
    return _lib.JointDesc(B, T, U, H, V, int(blank), _PREC[precision],
                          C.c_void_p(torch.cuda.current_stream().cuda_stream).value, int(tile_bound or 0), 1 if keep else 0)


def _workspace(desc, device):
    sz = C.c_size_t(0)
    _lib.check(_lib.load().rnntb200_joint_workspace_size(C.byref(desc), C.byref(sz)), "rnntb200_joint_workspace_size")
    return torch.empty(sz.value, dtype=torch.uint8, device=device)


def _check(enc, pred, W, b, labels, input_lengths, label_lengths):
    for t, n in ((enc, "enc_acts"), (pred, "pred_acts"), (W, "W"), (b, "b")):
        if not t.is_cuda:
            raise RuntimeError("%s must be a CUDA tensor: rnnt_b200 has no CPU path" % n)
        if t.dtype != torch.float32:
            raise TypeError("%s must be torch.float32" % n)
    for t, n in ((labels, "labels"), (input_lengths, "input_lengths"), (label_lengths, "label_lengths")):
        if t.dtype != torch.int32:
            raise TypeError("%s must be torch.int32" % n)
        if not t.is_cuda:
            raise RuntimeError("%s must be a CUDA tensor (device-resident lengths/labels, warprnnt_op.cc:88-94)" % n)
    if enc.dim() != 3 or pred.dim() != 3 or W.dim() != 2 or b.dim() != 1:
        raise ValueError("expected enc (B,T,H), pred (B,U,H), W (H,V), b (V)")
    B, T, H = enc.shape
    if pred.shape[0] != B or pred.shape[2] != H or W.shape[0] != H or b.shape[0] != W.shape[1]:
        raise ValueError("inconsistent shapes")
    U = pred.shape[1]
    if labels.dim() != 2 or labels.shape[0] != B or (labels.shape[1] != U - 1 and U > 1):
        raise ValueError("labels must be (B, U-1)")
    if input_lengths.shape != (B,) or label_lengths.shape != (B,):
        raise ValueError("must have a length per example.")


class _JointRNNT(torch.autograd.Function):
    @staticmethod
    def forward(ctx, enc, pred, W, b, labels, input_lengths, label_lengths, blank, precision, compact, keep=None, valid_tiles=None):
        L = _lib.load()
        enc, pred, W, b = (t.contiguous() for t in (enc, pred, W, b))
        labels, input_lengths, label_lengths = (t.contiguous() for t in (labels, input_lengths, label_lengths))
        _check(enc, pred, W, b, labels, input_lengths, label_lengths)
        B, T, H = enc.shape
        U, V = pred.shape[1], W.shape[1]
        lab = labels if labels.numel() else torch.zeros(1, dtype=torch.int32, device=enc.device)
        with torch.cuda.device(enc.device):
            # a backward will follow: let the forward keep its softmax numerators / tanh outputs in the workspace
            keep = any(ctx.needs_input_grad[:4]) if keep is None else bool(keep)
            desc = _desc(B, T, U, H, V, blank, precision, keep, valid_tiles)
            ws = _workspace(desc, enc.device)
            costs = torch.empty(B, dtype=torch.float32, device=enc.device)
            st = L.rnntb200_joint_loss_forward(C.byref(desc), _ptr(enc), _ptr(pred), _ptr(W), _ptr(b), _ptr(lab),
                                               _ptr(label_lengths), _ptr(input_lengths), _ptr(costs), _ptr(ws))
        _lib.check(st, "rnntb200_joint_loss_forward")
        ctx.save_for_backward(enc, pred, W, b, lab, input_lengths, label_lengths)
        ctx.ws, ctx.dims, ctx.blank, ctx.precision, ctx.compact, ctx.keep = ws, (B, T, U, H, V), blank, precision, compact, keep
        ctx.valid_tiles = valid_tiles
        return costs

    @staticmethod
    def backward(ctx, grad_costs):
        L = _lib.load()
        enc, pred, W, b, lab, input_lengths, label_lengths = ctx.saved_tensors
        B, T, U, H, V = ctx.dims
        g = grad_costs.to(torch.float32).contiguous()
        d_enc, d_pred, dW, db = (torch.empty_like(t) for t in (enc, pred, W, b))
        with torch.cuda.device(enc.device):
            desc = _desc(B, T, U, H, V, ctx.blank, ctx.precision, ctx.keep, ctx.valid_tiles)
            st = L.rnntb200_joint_loss_backward(C.byref(desc), _ptr(enc), _ptr(pred), _ptr(W), _ptr(b), _ptr(lab),
                                                _ptr(label_lengths), _ptr(input_lengths), _ptr(g), _ptr(d_enc),
                                                _ptr(d_pred), _ptr(dW), _ptr(db), _ptr(ctx.ws))
        _lib.check(st, "rnntb200_joint_loss_backward")
        ctx.ws = None
        return d_enc, d_pred, dW, db, None, None, None, None, None, None, None, None


def joint_rnnt_loss(enc_acts, pred_acts, W, b, labels, input_lengths, label_lengths, blank=0, precision="bf16",
                    compact=True, keep_activations=None, valid_tiles=None):
    """Per-utterance RNN-T NLL (B,) of logits = tanh(enc_acts[:,:,None]+pred_acts[:,None]) @ W + b,
    differentiable w.r.t. enc_acts, pred_acts, W, b -- without ever materialising (B,T,U,V).
    precision: 'bf16' = the tensor-core path (tcgen05, 16-bit operands, fp32 accumulate) or 'fp32' (exact CUDA-core path).
    'bf16' takes any vocabulary size V >= 1 and joint width 1 <= H <= 768 (the kernels pad to multiples of 64 internally;
    the gradients come back in the shapes of the inputs); H > 768 raises -- use 'fp32'.
    compact: accepted for compatibility and ignored -- ragged batches are compacted on the device, the library never
    synchronises with the host.
    keep_activations: None = automatically when a gradient is required (the forward then leaves its softmax
    numerators (bf16, 2 bytes per logit) in the workspace and the backward is two fused GEMM kernels);
    False = nothing of size O(B*T*U*V) survives the forward call; the backward re-runs the projection chunk by chunk
    (one more tensor-core pass).
    valid_tiles: optional promise `valid_tile_count(host lengths)` (rnntb200JointDesc.valid_tile_bound): sizes the workspace
    for the batch's valid lattice tiles instead of the padded (T,U) lattice, so that large ragged batches stay one chunk and
    keep their numerators; a broken promise yields NaN costs and a device-side message, never an out-of-bounds write."""
    return _JointRNNT.apply(enc_acts, pred_acts, W, b, labels, input_lengths, label_lengths, blank, precision, compact,
                            keep_activations, valid_tiles)


def joint_logits(enc_acts, pred_acts, W, b):
    """model.py:158-166's literal output: logits (B,T,U,V) float32, materialised (not differentiable;
    use joint_rnnt_loss for training).  For callers that want the reference's tensor itself."""
    L = _lib.load()
    enc, pred, W, b = (t.contiguous() for t in (enc_acts, pred_acts, W, b))
    B, T, H = enc.shape
    U, V = pred.shape[1], W.shape[1]
    with torch.cuda.device(enc.device):
        desc = _desc(B, T, U, H, V, 0, "fp32")
        ws = _workspace(desc, enc.device)
        out = torch.empty(B, T, U, V, dtype=torch.float32, device=enc.device)
        st = L.rnntb200_joint_logits(C.byref(desc), _ptr(enc), _ptr(pred), _ptr(W), _ptr(b), _ptr(out), _ptr(ws))
    _lib.check(st, "rnntb200_joint_logits")
    return out


def joint_step(f, g, K1, b1, K2, b2, want_logits=True, want_best=False):
    """``rnntb200_joint_step``: logits (B,V) of ONE lattice cell per batch row, tanh((f+g) @ K1 + b1) @ K2 + b2, and/or
    its argmax + log-softmax value.  ``f``, ``g``: (B,P) float32 CUDA views whose last dimension is contiguous (row
    strides are passed through, so ``encoded[:, i, :]`` / ``pred_out[:, -1, :]`` are not copied).  Not differentiable
    (inference).  Returns (logits | None, best | None, best_logp | None)."""
    L = _lib.load()
    for t, n in ((f, "f"), (g, "g"), (K2, "K2")):
        if not t.is_cuda or t.dtype != torch.float32:
            raise TypeError("%s must be a float32 CUDA tensor (rnnt_b200 has no CPU path)" % n)
    if f.dim() != 2 or g.shape != f.shape or f.stride(1) != 1 or g.stride(1) != 1:
        raise ValueError("f and g must be (B,P) with a contiguous last dimension")
    B, P = f.shape
    K1c = K1.detach().contiguous() if K1 is not None else None
    K2c = K2.detach().contiguous()
    H, V = K2c.shape
    b1c = b1.detach().contiguous() if b1 is not None else None
    b2c = b2.detach().contiguous() if b2 is not None else None
    with torch.cuda.device(f.device):
        logits = torch.empty(B, V, dtype=torch.float32, device=f.device) if want_logits else None
        best = torch.empty(B, dtype=torch.int32, device=f.device) if want_best else None
        logp = torch.empty(B, dtype=torch.float32, device=f.device) if want_best else None
        st = L.rnntb200_joint_step(_ptr(f.detach()), f.stride(0), _ptr(g.detach()), g.stride(0), _ptr(K1c), _ptr(b1c), _ptr(K2c),
                                   _ptr(b2c), B, P, H, V, _ptr(logits), _ptr(best), _ptr(logp),
                                   C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(st, "rnntb200_joint_step")
    return logits, best, logp


class _Dense1(torch.autograd.Function):
    """Keras Dense-1 of the joint (model.py:162-163) on the UN-broadcast inputs: ``x (..., P) @ K1 (P,H) [+ b1]`` and its three
    gradients through ``rnntb200_dense1_forward / _backward`` (the library's own fp32 kernels; SURVEY 8 f1)."""

    @staticmethod
    def forward(ctx, x, K1, b1):
        L = _lib.load()
        if not x.is_cuda or x.dtype != torch.float32 or K1.dtype != torch.float32:
            raise TypeError("dense1: float32 CUDA tensors required (rnnt_b200 has no CPU path)")
        P, H = K1.shape
        if x.shape[-1] != P:
            raise ValueError("dense1: x (..., %d) against a (%d, %d) kernel" % (x.shape[-1], P, H))
        xc, Kc = x.detach().contiguous(), K1.detach().contiguous()
        bc = b1.detach().contiguous() if b1 is not None else None
        rows = xc.numel() // P
        with torch.cuda.device(x.device):
            out = torch.empty(*x.shape[:-1], H, dtype=torch.float32, device=x.device)
            st = L.rnntb200_dense1_forward(_ptr(xc), rows, P, _ptr(Kc), _ptr(bc), H, _ptr(out),
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream))
        _lib.check(st, "rnntb200_dense1_forward")
        ctx.save_for_backward(xc, Kc)
        ctx.has_bias = b1 is not None
        return out

    @staticmethod
    def backward(ctx, d_out):
        L = _lib.load()
        xc, Kc = ctx.saved_tensors
        P, H = Kc.shape
        rows = xc.numel() // P
        dA = d_out.contiguous()
        need_x, need_k, need_b = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.has_bias and ctx.needs_input_grad[2]
        with torch.cuda.device(xc.device):
            dX = torch.empty_like(xc) if need_x else None
            dK = torch.zeros_like(Kc) if need_k else None          # the entry accumulates
            db = torch.zeros(H, dtype=torch.float32, device=xc.device) if need_b else None
            st = L.rnntb200_dense1_backward(_ptr(xc), _ptr(dA), _ptr(Kc), rows, P, H, _ptr(dX), _ptr(dK), _ptr(db),
                                            C.c_void_p(torch.cuda.current_stream().cuda_stream))
        _lib.check(st, "rnntb200_dense1_backward")
        return dX, dK, db


def dense1(x, K1, b1=None):
    """``x @ K1 (+ b1)`` through the extension (differentiable in x, K1, b1)."""
    return _Dense1.apply(x, K1, b1)


class Joint(torch.nn.Module):
    """The joint network of model.py:158-166 with Keras-layout parameters:
    dense_1 kernel (P,H) + bias (H) with tanh, dense_2 kernel (H,V) + bias (V).

    ``forward(inp_enc, pred_outputs)`` returns the reference's logits tensor (drop-in for the Keras
    model output); ``loss(...)`` runs the fused path where that tensor never exists."""

    def __init__(self, proj_size, joint_net_size, vocab_size, precision="bf16", blank=0):
        super().__init__()
        self.kernel_1 = torch.nn.Parameter(torch.empty(proj_size, joint_net_size))
        self.bias_1 = torch.nn.Parameter(torch.zeros(joint_net_size))
        self.kernel_2 = torch.nn.Parameter(torch.empty(joint_net_size, vocab_size))
        self.bias_2 = torch.nn.Parameter(torch.zeros(vocab_size))
        torch.nn.init.xavier_uniform_(self.kernel_1)   # Keras Dense default glorot_uniform
        torch.nn.init.xavier_uniform_(self.kernel_2)
        self.precision, self.blank = precision, blank

    def hoist(self, inp_enc, pred_outputs):
        """Dense-1 is linear before its tanh, so it is applied to the (B,T,P) and (B,U,P) inputs instead of the (B,T,U,P)
        lattice (SURVEY 8 a2), by the extension's own kernels (`dense1`: rnntb200_dense1_forward / _backward, SURVEY 8 f1)."""
        return dense1(inp_enc, self.kernel_1, self.bias_1), dense1(pred_outputs, self.kernel_1, None)

    def forward(self, inp_enc, pred_outputs):
        enc_acts, pred_acts = self.hoist(inp_enc, pred_outputs)
        return joint_logits(enc_acts, pred_acts, self.kernel_2, self.bias_2)

    def step(self, f, g):
        """Greedy-decode joint, utils/decoding.py:6-18: ``joint(model, f, g)`` adds ``f`` (B,T,P) to the LAST
        prediction-network frame ``g[:, -1, :]`` and returns ``outputs[:, 0, 0, :]`` -- the (B,V) logits of frame 0.
        One launch of the library's decode kernel (both Dense layers fused, fp32)."""
        return joint_step(f[:, 0, :], g[:, -1, :], self.kernel_1, self.bias_1, self.kernel_2, self.bias_2)[0]

    def greedy_step(self, f, g):
        """The decode step of utils/decoding.py:69-78 in one launch: ``preds = log_softmax(joint(model, f, g))``,
        ``predicted_id = argmax(preds)``.  Returns (predicted_id (B,) int32, its log-probability (B,) float32); the
        (B,V) logits are not written at all."""
        _, best, logp = joint_step(f[:, 0, :], g[:, -1, :], self.kernel_1, self.bias_1, self.kernel_2, self.bias_2,
                                   want_logits=False, want_best=True)
        return best, logp

    def loss(self, inp_enc, pred_outputs, labels, input_lengths, label_lengths):
        enc_acts, pred_acts = self.hoist(inp_enc, pred_outputs)
        return joint_rnnt_loss(enc_acts, pred_acts, self.kernel_2, self.bias_2, labels, input_lengths, label_lengths,
                               self.blank, self.precision)


def get_fused_loss_fn(reduction_factor, joint):
    """utils/loss.get_loss_fn-shaped adapter for the fused path: the returned function takes the joint
    network's INPUTS in place of y_pred (run_rnnt.py:269-273 collapsed into one call)."""
    _lib.load()

    def _loss_fn(y_true, inp_enc, pred_outputs, spec_lengths, label_lengths):
        y_true = y_true.to(torch.int32).contiguous()
        enc_lengths = encoder_lengths(spec_lengths, reduction_factor).contiguous()
        return joint.loss(inp_enc, pred_outputs, y_true, enc_lengths, label_lengths.to(torch.int32).contiguous())

    return _loss_fn
