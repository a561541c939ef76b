/** \file rnnt_b200.h
 *  C ABI of librnnt_b200.so -- the B200-native (sm_100a) RNN-T loss hot path.
 *
 *  Part 1 is a drop-in for the warp-transducer C interface the reference application binds
 *  (reference: warp-transducer/include/rnnt.h:16-143, implemented in
 *  warp-transducer/src/rnnt_entrypoint.cpp:14-185): same symbol names, argument order, status
 *  codes and by-value options struct, so the reference's TensorFlow op
 *  (tensorflow_binding/src/warprnnt_op.cc:105-141) or PyTorch binding
 *  (pytorch_binding/src/binding.cpp:84-154) links against this library unchanged.
 *
 *  Part 2 adds the entry points the reference has no analogue for: the fused joint-network +
 *  loss path (model.py:158-166 -> utils/loss.py:24-36 -> warp-transducer) in which the
 *  (B,T,U,V) fp32 logits are never written to HBM.  They follow the same conventions: status enum,
 *  caller-owned device workspace sized by a pure function, explicit CUstream.  The Part 2 calls are
 *  stream-ordered: no device allocation, no host synchronisation and no read-back (the only host
 *  synchronisation in the library is the one the reference's contract mandates at the end of
 *  compute_rnnt_loss: costs are host memory, gpu_rnnt.h:209-213).  State kept by the library:
 *  a per-(device, kernel) flag that the >48 KB dynamic shared memory opt-in has been set
 *  (mutex-protected; any number of devices and host threads per process), the launch counter and the
 *  optional timing records of rnntb200_set_timing.
 *
 *  What reaches HBM on the tensor-core path (N = lattice cells, V vocabulary):
 *    keep_activations = 0  forward: lse + two log-probs per cell, alpha, beta (O(N) floats).  The backward
 *                          re-runs the projection per utterance chunk, leaving 2 bytes per logit (bf16 softmax
 *                          numerators relative to one fp32 reference per lattice row) in the workspace for the two
 *                          gradient GEMM kernels to consume; no (B,T,U,V) tensor is produced by the forward call.
 *    keep_activations = 1  the forward itself writes those numerators (one pass fewer on the tensor cores).
 *    In both modes the logit gradients, dZ and z = tanh(enc+pred) exist only in shared / tensor memory.
 *
 *  There is NO CPU implementation in this library: loc == RNNT_CPU returns
 *  RNNT_STATUS_EXECUTION_FAILED (and says so on stderr) instead of silently falling back.
 */
#pragma once

#ifdef __cplusplus
#include <cstddef>
extern "C" {
#else
#include <stddef.h>
#include <stdbool.h>
#endif

/* forward declaration of the CUDA typedef (rnnt.h:13) */
typedef struct CUstream_st* CUstream;

/* ------------------------------------------------------------------------------------------
 * Part 1 -- warp-transducer compatible surface
 * ------------------------------------------------------------------------------------------ */

/** rnnt.h:16-22 */
typedef enum {
    RNNT_STATUS_SUCCESS = 0,
    RNNT_STATUS_MEMOPS_FAILED = 1,
    RNNT_STATUS_INVALID_VALUE = 2,
    RNNT_STATUS_EXECUTION_FAILED = 3,
    RNNT_STATUS_UNKNOWN_ERROR = 4
} rnntStatus_t;

/** rnnt.h:33-36 */
typedef enum { RNNT_CPU = 0, RNNT_GPU = 1 } rnntComputeLocation;

/** rnnt.h:43-64 -- 32 bytes on x86-64, passed BY VALUE.  batch_first is ignored by the GPU
 *  path exactly as in the reference (rnnt_entrypoint.cpp:75-76 never forwards it). */
struct rnntOptions {
    rnntComputeLocation loc;
    unsigned int num_threads;
    CUstream stream;
    int blank_label;
    int maxT;
    int maxU;
    bool batch_first;
};
#ifndef __cplusplus
typedef struct rnntOptions rnntOptions;
#endif

/** rnnt.h:25 / rnnt_entrypoint.cpp:14-16 -- API version, returns 1. */
int get_warprnnt_version();

/** rnnt.h:31 / rnnt_entrypoint.cpp:18-35 -- same five strings. */
const char* rnntGetStatusString(rnntStatus_t status);

/** rnnt.h:138-142 / rnnt_entrypoint.cpp:96-128.
 *  gpu == false returns the reference's CPU figure B*4*maxT*maxU*dtype (kept for host-logic
 *  parity; this library never uses a CPU workspace).  gpu == true returns what THIS library
 *  needs for compute_rnnt_loss: B*(4*SK + maxT*maxU + 2)*dtype with SK = (maxT+maxU-1)*maxU
 *  (diagonal-major lp_blank / lp_label / alpha / beta planes, the lse plane and the two
 *  log-likelihood vectors) -- larger than the reference's B*(3*maxT*maxU+2)*dtype, which is
 *  why callers must size the workspace through this function, as the reference's bindings do
 *  (warprnnt_op.cc:105-128, binding.cpp:120-137). */
rnntStatus_t get_workspace_size(int maxT, int maxU, int minibatch, bool gpu, size_t* size_bytes,
                                size_t dtype_size
#ifdef __cplusplus
                                = sizeof(float)
#endif
);

/** rnnt.h:104-113 / rnnt_entrypoint.cpp:38-93, GPU semantics (gpu_rnnt.h:82-215):
 *  activations  device, raw logits (B,maxT,maxU,V) row-major, softmax done inside
 *  gradients    device, same shape, or NULL for forward-only; padded cells are written 0
 *  flat_labels  DEVICE int32 (B, maxU-1) row-major (warprnnt_op.cc:88-94,193-195)
 *  label_lengths, input_lengths  DEVICE int32 (B)
 *  costs        HOST float (B): copied back and negated after a stream synchronise, as
 *               gpu_rnnt.h:209-213 does.  (rnntb200_loss_device below keeps them on device.)
 *  workspace    device, get_workspace_size(..., gpu=true) bytes
 *  Limits: maxU <= 1024 (one thread per label position, same bound as gpu_rnnt.h:127).
 *  Errors: NULL / non-positive arguments -> RNNT_STATUS_INVALID_VALUE (rnnt_entrypoint.cpp:49-60);
 *  CUDA launch failure -> RNNT_STATUS_EXECUTION_FAILED; copy failure -> RNNT_STATUS_MEMOPS_FAILED;
 *  loc == RNNT_CPU -> RNNT_STATUS_EXECUTION_FAILED (no CPU fallback). */
rnntStatus_t compute_rnnt_loss(const float* const activations, float* gradients, const int* const flat_labels,
                               const int* const label_lengths, const int* const input_lengths, int alphabet_size,
                               int minibatch, float* costs, void* workspace, rnntOptions options);

/** rnnt.h:115-124 / rnnt_entrypoint.cpp:130-185 -- double-precision twin. */
rnntStatus_t compute_rnnt_loss_fp64(const double* const activations, double* gradients,
                                    const int* const flat_labels, const int* const label_lengths,
                                    const int* const input_lengths, int alphabet_size, int minibatch,
                                    double* costs, void* workspace, rnntOptions options);

/* ------------------------------------------------------------------------------------------
 * Part 2 -- B200 additions (no reference analogue; conventions as above)
 * ------------------------------------------------------------------------------------------ */

/** compute_rnnt_loss with DEVICE costs and no host synchronisation.  This is
 *  what the torch surface calls; replaces the D2H + cudaStreamSynchronize of gpu_rnnt.h:209-213.
 *  grad_scale: optional DEVICE float (B); when non-NULL gradients[b] are pre-multiplied by it
 *  (folds _RNNTLossGrad's grad_loss[:,None,None,None]*grads, warprnnt_tensorflow/__init__.py:37-42). */
rnntStatus_t rnntb200_loss_device(const float* activations, float* gradients, const int* flat_labels,
                                  const int* label_lengths, const int* input_lengths, const float* grad_scale,
                                  int alphabet_size, int minibatch, float* costs_device, void* workspace,
                                  rnntOptions options);

typedef enum {
    RNNTB200_FP32_EXACT = 0, /**< fp32 CUDA-core arithmetic; parity gate rtol 1e-4 (BASELINE C1/C2) */
    RNNTB200_BF16_TC = 1     /**< 16-bit operands on tcgen05 tensor cores, fp32 accumulate (BASELINE C3-C5): the forward
                                  projection runs on fp16 z / W (11-bit significands), the two gradient GEMMs on bf16.
                                  Any V >= 1 and 1 <= H <= 768: the kernels run the problem padded to Hp = ceil64(H),
                                  Vp = ceil64(V), padding that contributes exactly zero (zero W / enc / pred columns, bias
                                  -inf for v >= V); inputs and outputs keep their unpadded shapes */
} rnntb200Precision;

/** Problem descriptor of the fused joint + loss path (model.py:158-166 hoisted form, SURVEY 8a2):
 *    z[b,t,u,:]  = tanh(enc[b,t,:] + pred[b,u,:])            model.py:158-163
 *    logits      = z . W + bias,  W is (H,V) row-major        model.py:165-166
 *    costs[b]    = RNN-T NLL of logits[b] (softmax inside)    utils/loss.py:24-36
 *  RNNTB200_BF16_TC takes any V >= 1 and 1 <= H <= 768 (H > 768: RNNT_STATUS_INVALID_VALUE, use RNNTB200_FP32_EXACT).
 *  Its workspace is that of the padded problem (ceil64(H), ceil64(V)); when H % 64 != 0 it also holds zero-padded copies
 *  of enc and pred (written by the forward, read by the backward) and d_enc at the padded width. */
typedef struct {
    int B, maxT, maxU, H, V;
    int blank_label;
    int precision; /* rnntb200Precision */
    CUstream stream;
    /** 0: unknown.  N > 0: the caller promises that at most N of the batch's 16 x 8 lattice tiles intersect the valid lattice,
     *  N >= sum_b ceil(T_b / 16) * ceil((U_b + 1) / 8) with U_b = label_lengths[b] (a host-side sum over lengths the data
     *  loader has anyway).  The kept numerators are indexed by compact tile slots, but only the device knows how many tiles
     *  are valid (the library never synchronises with the host), so by default the workspace is sized for every tile of
     *  the padded (maxT, maxU) lattice and a batch whose padded numerators exceed 16 GiB is processed in utterance chunks,
     *  which rules keep_activations out.  With a bound the workspace holds N row blocks and the batch is one chunk.  If
     *  the promise is broken nothing is written out of bounds: the forward prints an error and returns NaN costs.
     *  (Round 1 had `allow_host_sync` here: same offset and type, 0 keeps the old behaviour.) */
    int valid_tile_bound;
    /** 0: nothing but lse / log-prob pairs / alpha / beta survives the forward; the backward re-runs the projection
     *  chunk by chunk.  1 (tensor-core path): the forward also leaves, in the workspace, the softmax numerators of
     *  every lattice cell as bf16 (2 bytes per logit) and one fp32 reference per lattice row; the backward then skips its own
     *  projection pass.  Set it when a backward call will follow; it is honoured only when the whole batch fits one
     *  workspace chunk (<= 16 GiB of numerators), otherwise (and for fp32) ignored.  Must have the same value in the
     *  forward and the backward call. */
    int keep_activations;
} rnntb200JointDesc;

/** Bytes of device workspace the forward/backward pair needs (pure function of the descriptor). */
rnntStatus_t rnntb200_joint_workspace_size(const rnntb200JointDesc* desc, size_t* size_bytes);

/** Forward: enc (B,maxT,H), pred (B,maxU,H), W (H,V), bias (V) fp32 device; labels (B,maxU-1),
 *  label_lengths (B), input_lengths (B) int32 device; costs (B) fp32 DEVICE.  Leaves lse, the
 *  cached log-prob pairs, alpha and beta in `workspace` for the backward call. */
rnntStatus_t rnntb200_joint_loss_forward(const rnntb200JointDesc* desc, const float* enc, const float* pred,
                                         const float* W, const float* bias, const int* labels,
                                         const int* label_lengths, const int* input_lengths, float* costs,
                                         void* workspace);

/** Backward through the loss and the joint (run_rnnt.py:284's tape.gradient for this path):
 *  grad_costs (B) device = d(total)/d(costs[b]) (1/B for run_rnnt.py:278);
 *  outputs d_enc (B,maxT,H), d_pred (B,maxU,H), dW (H,V), db (V): fp32 device, OVERWRITTEN.
 *  Must follow a forward call with the same descriptor, inputs and workspace. */
rnntStatus_t rnntb200_joint_loss_backward(const rnntb200JointDesc* desc, const float* enc, const float* pred,
                                          const float* W, const float* bias, const int* labels,
                                          const int* label_lengths, const int* input_lengths,
                                          const float* grad_costs, float* d_enc, float* d_pred, float* dW,
                                          float* db, void* workspace);

/** Joint network forward only, materialising logits (B,maxT,maxU,V) fp32 -- the literal
 *  model.py:158-166 output, used by the drop-in `Joint` module when a caller wants the tensor
 *  (e.g. to feed rnnt_loss/compute_rnnt_loss exactly as run_rnnt.py:269-273 does). */
rnntStatus_t rnntb200_joint_logits(const rnntb200JointDesc* desc, const float* enc, const float* pred,
                                   const float* W, const float* bias, float* logits, void* workspace);

/** Greedy-decode joint (utils/decoding.py:6-18, called per step at :69-78): one lattice cell per batch row,
 *    logits[b,:] = tanh((f[b,:] + g[b,:]) . K1 + b1) . K2 + b2;  best[b] = argmax_v logits (smallest index among equal
 *    maxima, as tf.argmax);  best_logp[b] = log_softmax(logits[b])[best[b]]
 *  in ONE launch (thread-block clusters of 8 CTAs per row; fp32 FMA arithmetic).  f, g: (B,P) device rows with strides
 *  ldf, ldg (so f = encoded[:, i, :] and g = pred_out[:, -1, :] need no copy); K1 (P,H) and b1 (H) are Keras Dense-1
 *  (K1 == NULL: f, g are the already projected activations, P == H); K2 (H,V), b2 (V).  Any of logits (B,V), best (B),
 *  best_logp (B) may be NULL, not all.  P <= 4096, H <= 2048. */
rnntStatus_t rnntb200_joint_step(const float* f, long long ldf, const float* g, long long ldg, const float* K1,
                                 const float* b1, const float* K2, const float* b2, int B, int P, int H, int V,
                                 float* logits, int* best, float* best_logp, CUstream stream);

/** Dense-1 of the joint (model.py:162-163, Keras kernel (P,H) + bias (H)) applied BEFORE the broadcast add -- it is linear in
 *  front of its tanh, so W1^T (f_t + g_u) + b1 = (W1^T f_t + b1) + W1^T g_u (SURVEY 8 a2): the hot path's inputs
 *  enc_acts / pred_acts are these two projections.
 *    forward:   out[r,:] = X[r,:] . K1 (+ b1)                       X (rows,P) -> out (rows,H), b1 may be NULL (the pred side)
 *    backward:  dX = dA . K1^T;  dK1 += X^T . dA;  db1 += sum_r dA[r,:]      (dX, dK1, db1 may each be NULL; dK1 / db1 are
 *               ACCUMULATED into, so the encoder-side and the prediction-side call add into one zeroed buffer)
 *  fp32 FMA kernels of this library (no GEMM library).  dK1 is a split-K product combined with float atomics: its last bits
 *  depend on the order the partial sums arrive in (as the exact fp32 path's dW). */
rnntStatus_t rnntb200_dense1_forward(const float* X, long long rows, int P, const float* K1, const float* b1, int H,
                                     float* out, CUstream stream);
rnntStatus_t rnntb200_dense1_backward(const float* X, const float* dA, const float* K1, long long rows, int P, int H,
                                      float* dX, float* dK1, float* db1, CUstream stream);

/** Number of kernels launched by this library in this process since load (bench.py's gpu_launches).  Every kernel
 *  on the path is the library's own: it links no GEMM library. */
unsigned long long rnntb200_launch_count();

/** Per-kernel CUDA-event instrumentation for bench.py's attribution pass.  set_timing(1) clears the record
 *  list and enables recording (events on the launching stream around each hot kernel); set_timing(0)
 *  disables and clears.  After synchronising the stream, get_timing(i, &name, &ms) returns 1 and the i-th
 *  record, or 0 past the end.  Off by default; never enabled inside a timed benchmark region. */
void rnntb200_set_timing(int on);
int rnntb200_get_timing(int index, const char** name, float* ms);

/** Build info string: "rnnt_b200 <version> sm_100a tcgen05=<0|1>". */
const char* rnntb200_build_info();

#ifdef __cplusplus
}
#endif
