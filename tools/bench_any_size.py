"""Step time of the fused joint + loss (forward + backward) at vocabulary sizes and joint widths that are not multiples of 64,
against their aligned padded twins and against the fp32 CUDA-core path -- the only option those shapes had before the
tensor-core kernels learnt to pad internally.

    python tools/bench_any_size.py [--steps 20] [--warmup 3] [--out FILE.json]

Geometry of BASELINE C3 (B=32, T=512, U=128, full lengths).  All configurations live in one process and are timed
round-robin, one step of each per round (the order rotates every round), with CUDA events around each step; the JSON
reports per configuration the median, minimum and 90th percentile over the timed steps, and per comparison the ratio of
medians.  The card's name and power limit are read in the same run (nvidia-smi), since they are part of every number.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

B, T, U = 32, 512, 128

# (name, H, V, precision)
CONFIGS = [
    ("H640_V1024", 640, 1024, "bf16"),
    ("H640_V1025", 640, 1025, "bf16"),
    ("H640_V1088", 640, 1088, "bf16"),
    ("H600_V1024", 600, 1024, "bf16"),
    ("H640_V31", 640, 31, "bf16"),
    ("H640_V64", 640, 64, "bf16"),
    ("H640_V31_fp32", 640, 31, "fp32"),
    ("H640_V4073", 640, 4073, "bf16"),
    ("H640_V4096", 640, 4096, "bf16"),
    ("H640_V4073_fp32", 640, 4073, "fp32"),
]
# (what, configuration, against)
COMPARISONS = [
    ("V=1025 vs its padded twin V=1088", "H640_V1025", "H640_V1088"),
    ("V=1025 vs V=1024", "H640_V1025", "H640_V1024"),
    ("H=600 vs its padded twin H=640", "H600_V1024", "H640_V1024"),
    ("V=31 vs its padded twin V=64", "H640_V31", "H640_V64"),
    ("V=31 bf16 vs fp32", "H640_V31", "H640_V31_fp32"),
    ("V=4073 vs its padded twin V=4096", "H640_V4073", "H640_V4096"),
    ("V=4073 bf16 vs fp32", "H640_V4073", "H640_V4073_fp32"),
]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        dev = torch.cuda.current_device()
        name, power = (x.strip() for x in out[dev].split(","))
        return {"name": name, "power_limit": power}
    except Exception as e:    # the figures stay usable, but say that the card could not be identified
        return {"name": torch.cuda.get_device_name(), "power_limit": "unknown (%s)" % type(e).__name__}


def make_inputs(H, V, gen):
    dev = "cuda"
    t = dict(enc=torch.randn(B, T, H, device=dev, generator=gen), pred=torch.randn(B, U, H, device=dev, generator=gen),
             W=torch.randn(H, V, device=dev, generator=gen) / H ** 0.5, b=0.1 * torch.randn(V, device=dev, generator=gen))
    for x in t.values():
        x.requires_grad_()
    t["labels"] = torch.randint(1, max(V, 2), (B, U - 1), dtype=torch.int32, device=dev, generator=gen)
    t["il"] = torch.full((B,), T, dtype=torch.int32, device=dev)
    t["ll"] = torch.full((B,), U - 1, dtype=torch.int32, device=dev)
    return t


def step(rb, t, precision):
    for n in ("enc", "pred", "W", "b"):
        t[n].grad = None
    costs = rb.joint_rnnt_loss(t["enc"], t["pred"], t["W"], t["b"], t["labels"], t["il"], t["ll"], precision=precision)
    (costs.sum() / B).backward()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--only", default="", help="comma-separated configuration names (default: all)")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    import rnnt_speech_recognition_b200 as rb
    torch.backends.cuda.matmul.allow_tf32 = False
    cfgs = [c for c in CONFIGS if not args.only or c[0] in args.only.split(",")]
    gen = torch.Generator(device="cuda")
    gen.manual_seed(0)
    inputs = {c[0]: make_inputs(c[1], c[2], gen) for c in cfgs}
    for _ in range(args.warmup):
        for name, H, V, prec in cfgs:
            step(rb, inputs[name], prec)
    torch.cuda.synchronize()
    times = {c[0]: [] for c in cfgs}
    for r in range(args.steps):
        order = cfgs[r % len(cfgs):] + cfgs[:r % len(cfgs)]
        ev = []
        for name, H, V, prec in order:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step(rb, inputs[name], prec)
            b.record()
            ev.append((name, a, b))
        torch.cuda.synchronize()
        for name, a, b in ev:
            times[name].append(a.elapsed_time(b))
    res = {"gpu": gpu_info(), "geometry": {"B": B, "T": T, "U": U}, "steps": args.steps, "warmup": args.warmup,
           "torch": torch.__version__, "configs": {}, "comparisons": []}
    for name, H, V, prec in cfgs:
        x = np.array(times[name])
        res["configs"][name] = {"H": H, "V": V, "precision": prec, "ms_median": float(np.median(x)), "ms_min": float(x.min()),
                                "ms_p90": float(np.percentile(x, 90))}
    for what, a, b in COMPARISONS:
        if a in res["configs"] and b in res["configs"]:
            res["comparisons"].append({"what": what, "ratio_of_medians": res["configs"][a]["ms_median"] / res["configs"][b]["ms_median"]})
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
