#!/usr/bin/env python
"""bench.py -- RNN-T loss+grad utterances/sec (BASELINE.json metric) on N B200s of one node.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path on the host cores
  python bench.py ... --dump-outputs DIR                    # also saves the last timed step's outputs, to compare builds

A "step" is one pass of the hot path (joint forward -> alpha/beta -> gradients to enc_acts, pred_acts,
W, b) over one synthetic batch of the BASELINE C3 shape (B=32,T=512,U=128,V=1024,H=640 per GPU, bf16
tensor-core path; --workload c2 runs the fp32 C2 shape).  Default = weak scaling: every rank holds a full
batch; --scaling strong = BASELINE C4 literally (ONE global batch of B utterances sharded over the ranks, 4 per GPU at
N=8).  An N>1 weak run also measures the strong point and reports it under "strong".  The only collective is ONE
packed all-reduce of [loss_sum | dW | db] per step.

Printed JSON (one line, rank 0): see the task contract -- value (inputs resident in HBM), e2e (host
buffers through the public torch API, H2D/D2H inside the timed region), roofline of the dominant
kernel (CUDA events on the launching stream, attribution pass outside the timed region),
cpu_baseline (reference library + torch-CPU joint on the host cores), clocks, gpu_launches.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the source tree (it may be read-only)

WORKLOADS = {
    "c3": dict(B=32, T=512, U=128, V=1024, H=640, precision="bf16", dtype="bf16"),
    "c2": dict(B=16, T=256, U=64, V=256, H=320, precision="fp32", dtype="f32"),
    "c1": dict(B=2, T=20, U=8, V=32, H=64, precision="fp32", dtype="f32"),
    # BASELINE C5: Common-Voice-shaped ragged batch (SURVEY 8d: seed 1234, T_b ~ U{100..1600}, U_b ~ U{10..200},
    # one utterance forced to (1600,200) and one to (100,10)); padded/masked lattice stress
    "c5": dict(B=64, T=1600, U=200, V=4096, H=640, precision="bf16", dtype="bf16", ragged=True),
}
METRIC = "rnnt_loss_grad_utterances_per_sec"
# what one step hands its caller, in the order step() returns it
OUTPUT_NAMES = ("loss", "costs", "d_enc", "d_pred", "dW", "db")
DUMP_BYTES = 64 * 10 ** 6              # all files of --dump-outputs together


def dump_sample(named):
    """{name: float32 numpy array} of the device tensors in `named`: whole when together they fit DUMP_BYTES; otherwise the
    larger ones are cut to a fixed, seeded sample of their flattened elements (in index order) so that the total fits.
    The sample depends on the shapes only, so two runs with the same arguments dump the same elements."""
    import numpy as np
    import torch
    sizes = {n: t.numel() for n, t in named.items()}
    left, out = (DUMP_BYTES - 1024 * len(named)) // 4, {}            # 1 KiB per file for the .npy header
    for i, n in enumerate(sorted(sizes, key=sizes.get)):
        keep = min(sizes[n], left // (len(sizes) - i))
        left -= keep
        t = named[n].detach().float()
        if keep < sizes[n]:
            idx = np.sort(np.random.default_rng(0).choice(sizes[n], keep, replace=False, shuffle=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        out[n] = t.cpu().numpy()
    return out


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def csrc_sha16():
    """Hash of the CUDA sources: an ncu capture is only quoted next to a number when it was taken from THIS source."""
    import glob
    import hashlib
    h = hashlib.sha256()
    for f in sorted(glob.glob(os.path.join(ROOT, "rnnt_speech_recognition_b200", "csrc", "*.cu*"))):
        h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


def measured_traffic():
    """profiles/rNN/traffic.json = {"csrc_sha16": ..., "kernels": {name: dram bytes per launch}, "step": bytes} written by
    tools/ncu_summary.py from an `ncu --set full` capture.  Returned only if it was captured from the current sources
    (otherwise the figure would silently go stale the moment a kernel changes)."""
    import glob
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*", "traffic.json")), reverse=True):
        try:
            t = json.load(open(f))
            if t.get("csrc_sha16") == csrc_sha16():
                t["file"] = os.path.relpath(f, ROOT)
                return t
        except Exception:
            pass
    return None


def synth(cfg, seed, device, pin=False):
    import torch
    g = torch.Generator().manual_seed(seed)
    B, T, U, V, H = (cfg[k] for k in "BTUVH")
    d = dict(enc=torch.randn(B, T, H, generator=g), pred=torch.randn(B, U, H, generator=g),
             W=torch.randn(H, V, generator=g) / H ** 0.5, b=torch.zeros(V),
             labels=torch.randint(1, V, (B, U - 1), generator=g, dtype=torch.int32),
             il=torch.full((B,), T, dtype=torch.int32), ll=torch.full((B,), U - 1, dtype=torch.int32))
    if cfg.get("ragged"):
        d["il"] = torch.randint(100, T + 1, (B,), generator=g, dtype=torch.int32)
        d["ll"] = torch.randint(10, U + 1, (B,), generator=g, dtype=torch.int32) - 1
        d["il"][0], d["ll"][0] = T, U - 1
        d["il"][1], d["ll"][1] = 100, 9
        for i in range(B):
            d["enc"][i, d["il"][i]:] = 0
            d["pred"][i, d["ll"][i] + 1:] = 0
            d["labels"][i, d["ll"][i]:] = 0
    if pin:
        return {k: v.pin_memory() for k, v in d.items()}
    return {k: v.to(device) for k, v in d.items()}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([x.strip() for x in line.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = []
        for i, n in ((4, "hw_slowdown"), (5, "hw_thermal_slowdown"), (6, "sw_thermal_slowdown"), (7, "sw_power_cap")):
            if any(len(r) >= 8 and r[i].lower().startswith("active") for r in self.rows):
                reasons.append(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own CPU implementation of the path on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_reference_runner(cfg):
    """Returns (run(n_utts) -> seconds, kind, cores, note).  What run_rnnt.py executes on a CPU-only
    TF build: joint forward (model.py:158-166) -> log_softmax (utils/loss.py:29-30) ->
    compute_rnnt_loss(RNNT_CPU) -> backward to d_enc, d_pred, dW, db.  The loss library is the
    UNMODIFIED reference (oracle/_ref/libwarprnnt.so) when it was built; TensorFlow 2.2 is not
    installable here, so the Dense/tanh/log_softmax/autograd pieces run as torch-CPU fp32 ops on all
    host threads.  Without oracle/_ref the C oracle port (oracle/rnnt_oracle.c) stands in."""
    import numpy as np
    import torch
    from oracle import oracle
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    B, T, U, V, H = (cfg[k] for k in "BTUVH")
    d = synth(cfg, 1234, "cpu")
    # micro-batch of the CPU arm: 4 utterances (BASELINE.md section 4) unless their (mb,T,U,V) fp32 slabs -- logits, log-probs,
    # gradients and their autograd copies -- would not fit a host comfortably (C5: 5.2 GB per utterance and slab)
    mb_default = max(1, min(4, int(6e9 // (4.0 * T * U * V))))
    if oracle.have_ref():
        class RefLoss(torch.autograd.Function):
            @staticmethod
            def forward(ctx, lp, labels, il, ll):
                costs, grads = oracle.ref_cpu_cost_and_grad(lp.detach().numpy(), labels, il, ll, num_threads=cores)
                ctx.grads = torch.from_numpy(grads)
                return torch.from_numpy(costs)

            @staticmethod
            def backward(ctx, go):
                return ctx.grads.mul_(go.view(-1, 1, 1, 1)), None, None, None

        def run(n, mb=mb_default):
            # micro-batches of `mb` utterances (BASELINE.md section 4): utterances are independent (cpu_rnnt.h:290-301) and
            # warp-transducer's OpenMP loop parallelises over the minibatch only, so a micro-batch gives it work while the
            # (mb,T,U,V) slabs stay a few GB
            t0 = time.perf_counter()
            W, b = d["W"].clone().requires_grad_(), d["b"].clone().requires_grad_()
            for i0 in range(0, n, mb):
                j = [(i0 + k) % B for k in range(min(mb, n - i0))]
                e, p = d["enc"][j].clone().requires_grad_(), d["pred"][j].clone().requires_grad_()
                z = torch.tanh(e[:, :, None, :] + p[:, None, :, :])
                lp = torch.log_softmax(z @ W + b, -1)
                c = RefLoss.apply(lp, d["labels"][j].numpy(), d["il"][j].numpy(), d["ll"][j].numpy())
                (c.sum() / B).backward()
            return time.perf_counter() - t0
        return run, "reference", cores, mb_default, ("oracle/_ref/libwarprnnt.so (unmodified reference, OpenMP over the micro-batch) + "
                                                     "torch-CPU fp32 joint/autograd, micro-batches of %d utterance(s)" % mb_default)

    a = {k: v.numpy() for k, v in d.items()}

    def run(n, mb=mb_default):
        t0 = time.perf_counter()
        idx = [i % B for i in range(n)]
        oracle.joint_loss_grad(a["enc"][idx], a["pred"][idx], a["W"], a["b"], a["labels"][idx], a["il"][idx],
                               a["ll"][idx], grad_scale=np.full(n, 1.0 / B, np.float32))
        return time.perf_counter() - t0
    return run, "port", cores, mb_default, "oracle/rnnt_oracle.c (C restatement, OpenMP)"


def cpu_baseline(cfg, budget_s=20.0):
    run, kind, cores, mb, note = cpu_reference_runner(cfg)
    t1 = run(1)                                     # warm-up + calibration
    n = max(1, min(cfg["B"], mb * max(1, int(budget_s / 3 / max(mb * t1, 1e-3)))))   # whole micro-batches
    reps = max(1, min(3, int(budget_s / max(n * t1, 1e-3))))
    ts = [run(n) for _ in range(reps)]              # best of up to 3 (BASELINE.md section 4)
    t = min(ts)
    return {"value": n / t, "unit": "utt/s", "cores": cores, "kind": kind,
            "sample": "%d utterance(s) of the workload shape, best of %d runs (%.1f s each); %s" % (n, reps, t, note)}


def reference_arm(args, cfg, rank):
    if rank != 0:
        return
    run, kind, cores, mb, note = cpu_reference_runner(cfg)
    t1 = run(1)
    total = args.steps + args.warmup
    n = max(1, min(cfg["B"], int(150.0 / (total * max(t1, 1e-3)))))
    if n >= mb:
        n -= n % mb                                 # whole micro-batches
    for _ in range(args.warmup):
        run(n)
    times = [run(n) for _ in range(args.steps)]
    tot = sum(times)
    val = n * args.steps / tot
    sample = "%d utterance(s) per step; %s" % (n, note)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "utt/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(cfg, args.gpus, args.workload, args.scaling),
        "cpu_baseline": {"value": val, "unit": "utt/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def workload_config(cfg, n_gpus, name, scaling="weak"):
    strong = scaling == "strong"
    return {"workload": "BASELINE %s: B=%d T=%d U=%d V=%d H=%d %s%s, joint fwd + alpha/beta + grads (d_enc,d_pred,dW,db)"
                        % (name.upper(), cfg["B"], cfg["T"], cfg["U"], cfg["V"], cfg["H"],
                           "GLOBAL batch sharded over the GPUs" if strong else "per GPU",
                           " (ragged T_b in [100,T], U_b in [10,U])" if cfg.get("ragged") else ""),
            "global_batch": cfg["B"] * (1 if strong else n_gpus), "parallelism": "dp%d" % n_gpus, "precision": cfg["precision"],
            "l2": "256 MiB scratch write between timed steps; per-step working set (>4 GB) exceeds the 126 MB L2"}


def op_path_block(pk):
    """Materialised-logits entry (compute_rnnt_loss, the warp-transducer-compatible C ABI) on this GPU: ms per call,
    achieved GB/s on SURVEY 8(d)'s algorithmic bytes 3*N*V*4 + 24*N against the measured HBM peak, and the reference's
    own SIMT kernels (oracle/_ref/libwarprnnt_gpu.so, compiled unmodified for sm_100) on the same inputs."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import bench_op
        out = []
        for r in bench_op.run_shapes([(16, 256, 64, 256), (32, 512, 128, 1024)]):
            r["frac_of_hbm_peak"] = r["rnnt_b200"]["GBps"] / pk["hbm_gbs"]
            out.append(r)
        return out
    except Exception as e:                      # never let the secondary block take the headline line down
        return {"error": repr(e)}


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-op-path", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (%s) to DIR/<name>.npy as float32, at most %d MB in "
                         "all: beyond that the larger arrays become a fixed, seeded sample of their flattened elements; "
                         "rank 0 only" % (", ".join(OUTPUT_NAMES), DUMP_BYTES // 10 ** 6))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    cfg = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, cfg, rank)
        return

    import torch
    import torch.distributed as dist
    import rnnt_speech_recognition_b200 as rb
    from rnnt_speech_recognition_b200 import _lib, distributed as D
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries ONE JSON line.  NCCL prints its version banner (NCCL_DEBUG=VERSION on the GPU boxes) with a plain
    # printf, so file descriptor 1 is pointed at stderr for the whole run and the result line is written to the saved
    # descriptor at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, T, U, V, H = (cfg[k] for k in "BTUVH")

    def shard(full, scaling):
        """weak: this rank's own batch of B; strong: its contiguous shard of ONE global batch of B (run_rnnt.py:87-88)."""
        if scaling == "weak":
            return full, B * world
        lo, hi = D.shard_bounds(B, world, rank)
        return {k: (v[lo:hi].contiguous() if k in ("enc", "pred", "labels", "il", "ll") else v) for k, v in full.items()}, B

    full_dev = synth(cfg, 1234 + (rank if args.scaling == "weak" else 0), dev)
    d, gB = shard(full_dev, args.scaling)
    host_full = synth(cfg, 1234 + (rank if args.scaling == "weak" else 0), dev, pin=True)
    host = shard(host_full, args.scaling)[0]
    host = {k: (v.pin_memory() if not v.is_pinned() else v) for k, v in host.items()}
    params = [full_dev["W"].clone().requires_grad_(), full_dev["b"].clone().requires_grad_()]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    # what a data loader knows on the host: how many 16 x 8 lattice tiles of the batch are valid.  Lets a ragged batch whose
    # PADDED numerators exceed one workspace chunk (C5) stay one chunk and keep them; ignored for batches that fit anyway (C3)
    mode = {"keep": None, "gB": gB, "vt": rb.valid_tile_count(host["il"].tolist(), host["ll"].tolist())}

    def step(enc, pred, labels, il, ll):
        enc.requires_grad_(), pred.requires_grad_()
        for p in params:
            p.grad = None
        costs = rb.joint_rnnt_loss(enc, pred, params[0], params[1], labels, il, ll, precision=cfg["precision"],
                                   keep_activations=mode["keep"], valid_tiles=mode["vt"])
        loss_sum = costs.sum()
        (loss_sum / mode["gB"]).backward()                           # run_rnnt.py:278
        ls, dW, db = D.allreduce_loss_and_weight_grads(loss_sum.detach(), params[0].grad, params[1].grad)
        return ls / mode["gB"], costs.detach(), enc.grad, pred.grad, dW, db          # OUTPUT_NAMES

    cur = {"d": d}

    def resident_step():
        x = cur["d"]
        return step(x["enc"].detach(), x["pred"].detach(), x["labels"], x["il"], x["ll"])

    # e2e: every step copies ITS inputs from pinned host memory and reads its loss back.  The copy of step i+1 is
    # issued on a copy stream while step i computes (what a prefetching input pipeline does); the compute stream
    # waits on the copy's event, and the tensors are handed over with record_stream.
    copy_stream = torch.cuda.Stream(device=dev)
    pending = {}

    def issue_copy():
        with torch.cuda.stream(copy_stream):
            dd = {k: host[k].to(dev, non_blocking=True) for k in ("enc", "pred", "labels", "il", "ll")}
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        pending["next"] = (dd, ev)

    def e2e_step():
        if "next" not in pending:
            issue_copy()
        dd, ev = pending.pop("next")
        torch.cuda.current_stream().wait_event(ev)
        for v in dd.values():
            v.record_stream(torch.cuda.current_stream())
        issue_copy()                                                  # next step's H2D overlaps this step's kernels
        out = step(dd["enc"], dd["pred"], dd["labels"], dd["il"], dd["ll"])
        return out[0].item()                                          # D2H read of the step's loss

    def timed(fn, steps, keep=None):
        """Milliseconds of `steps` calls of fn.  keep: a dict that receives what the LAST call returned; every other call's
        result is dropped at once, as a caller's would be, so that no step holds its predecessor's outputs in memory."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        for i, (a, b) in enumerate(ev):
            flush.zero_()                                             # L2 flush, outside the event pair
            a.record()
            if keep is None or i + 1 < steps:
                fn()
            else:
                keep["out"] = fn()
            b.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)                 # max over ranks
        return ms.item()

    for _ in range(args.warmup):
        resident_step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = _lib.launch_count()
    last = {} if args.dump_outputs and rank == 0 else None
    ms = timed(resident_step, args.steps, keep=last)
    launches = _lib.launch_count() - l0
    dumped = dump_sample(dict(zip(OUTPUT_NAMES, last.pop("out")))) if last is not None else None
    for _ in range(2):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    # the same step with NOTHING of size O(N*V) surviving the forward call (keep_activations = 0: the backward re-runs
    # the projection chunk by chunk) -- the north-star-literal mode, reported beside the default
    ms_nomat = None
    if cfg["precision"] == "bf16":
        mode["keep"] = False
        for _ in range(2):
            resident_step()
        ms_nomat = timed(resident_step, args.steps)
        mode["keep"] = None
    # N > 1, weak run: also the BASELINE C4 strong-scaling point (one global batch of B sharded over the ranks)
    strong = None
    if world > 1 and args.scaling == "weak" and B >= world:
        sd, sgB = shard(synth(cfg, 1234, dev), "strong")
        cur["d"], mode["gB"] = sd, sgB
        mode["vt"] = rb.valid_tile_count(sd["il"].tolist(), sd["ll"].tolist())
        for _ in range(3):
            resident_step()
        ms_s = timed(resident_step, args.steps)
        strong = {"value": sgB * args.steps / (ms_s * 1e-3), "unit": "utt/s", "ms_per_step": ms_s / args.steps,
                  "global_batch": sgB, "utt_per_gpu": sgB / world, "scaling": "strong",
                  "note": "BASELINE C4: B=%d sharded over %d GPUs, same step, max over ranks" % (sgB, world)}
        cur["d"], mode["gB"] = d, gB
    if sampler:
        sampler.stop_flag.set()
        sampler.join(timeout=3)

    # attribution pass (outside every timed region): per-kernel CUDA-event durations on the launching stream
    kernels = {}
    _lib.set_timing(True)
    resident_step()
    torch.cuda.synchronize()
    for name, t in _lib.get_timings():
        kernels[name] = kernels.get(name, 0.0) + t
    _lib.set_timing(False)

    if rank == 0:
        pk, pk_src = peaks()
        N = int((d["il"].long() * (d["ll"].long() + 1)).sum().item())      # valid lattice cells of this rank (== B*T*U when not ragged)
        traffic = measured_traffic()
        if cfg["precision"] == "bf16":
            flops = 2.0 * N * H * V
            dom = next((k for k in kernels if k.endswith("<fwd>") or k.endswith("<fwd+keep>")), "joint_tc3_kernel<fwd+keep>")
            t_dom = kernels.get(dom)
            ach = flops / (t_dom * 1e-3) / 1e12 if t_dom else None
            peak = pk["bf16_tflops_sustained"]
            roof = {"kernel": dom, "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                    "frac": (ach / peak) if ach else None,
                    "traffic": (traffic or {}).get("kernels", {}).get(dom),
                    "peak_source": "%s bf16 sustained (kernel timed inside the step)" % pk_src,
                    "algorithmic_flops_per_launch": flops, "launch_ms": t_dom,
                    "step": {"algorithmic_flops": 6.0 * N * H * V,
                             "achieved": 6.0 * N * H * V / (ms / args.steps * 1e-3) / 1e12,
                             "frac": 6.0 * N * H * V / (ms / args.steps * 1e-3) / 1e12 / peak}}
        else:
            dom = "alpha_beta_kernel"
            t_dom = kernels.get(dom)
            byts = 24.0 * N
            ach = byts / (t_dom * 1e-3) / 1e9 if t_dom else None
            roof = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": (ach / pk["hbm_gbs"]) if ach else None,
                    "traffic": (traffic or {}).get("kernels", {}).get(dom), "peak_source": pk_src,
                    "algorithmic_bytes_per_launch": byts, "launch_ms": t_dom}
        h2d = sum(host[k].numel() * host[k].element_size() for k in ("enc", "pred", "labels", "il", "ll"))
        out = {
            "metric": METRIC, "value": gB * args.steps / (ms * 1e-3), "unit": "utt/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic",
            "config": workload_config(cfg, world, args.workload, args.scaling),
            "clocks": sampler.summary() if sampler else None,
            "e2e": {"value": gB * args.steps / (ms_e2e * 1e-3), "unit": "utt/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps,
                    "note": "inputs in (enc, pred, labels, lengths from pinned host memory), loss out (4 B); the gradients "
                            "(d_enc, d_pred, dW, db) stay on the device where the optimizer / upstream autograd consumes them"},
            "gpu_launches": int(launches), "roofline": roof,
            "kernels_ms": {k: round(v, 4) for k, v in sorted(kernels.items(), key=lambda kv: -kv[1])},
        }
        if ms_nomat is not None:
            out["value_no_materialise"] = {"value": gB * args.steps / (ms_nomat * 1e-3), "unit": "utt/s",
                                           "ms_per_step": ms_nomat / args.steps,
                                           "note": "keep_activations=0: nothing of size O(N*V) survives the forward call; "
                                                   "`value` is the default mode (forward keeps 2 B per logit for the backward)"}
        out["dram_bytes_per_step"] = ({"value": traffic.get("step"), "source": traffic["file"] + " (ncu --set full of this "
                                       "source tree, csrc_sha16 %s)" % traffic["csrc_sha16"]} if traffic else None)
        if strong:
            out["strong"] = strong
        if world == 1 and not args.no_op_path and args.workload == "c3":
            out["op_path"] = op_path_block(pk)
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(cfg, args.cpu_budget)
        if dumped:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for n, a in dumped.items():
                np.save(os.path.join(args.dump_outputs, n + ".npy"), a)
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
