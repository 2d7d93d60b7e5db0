"""bf16 logits through the flat step (FusedFlatStep, flat7_620_b4: B = 4, 620 x 620, K = 7), one JSON line.

Three arms, each a full step (forward + the gradient reaching the logits) captured in a CUDA graph:
  fp32        fp32 logits into the step;
  workaround  bf16 logits cast with .float() into the fp32 step, the gradient cast back to bf16 by autograd (what a user
              had to write before the step read bf16);
  bf16        bf16 logits into the step (RHSEG_LOGITS_BF16).
Inputs: bench.synth_inputs (seed 1000, drawn on the GPU).  Before timing, the bf16 step is checked against the fp32 step
on the upcast logits (the bounds of tests/test_gpu_flat_bf16.py).  Timing follows tools/bench_bf16.py: warmed graphs,
alternating blocks of replays (>= --min-ms of timed work per arm), the median block reported.  Also per arm: the peak
memory one eager step allocates above its inputs, and the device launches (kernels, memsets, copies) of one eager step
(torch.profiler, after timing).  --arms fp32 times the fp32 arm alone (an A/B of two builds through RHSEG_LIB).
    python tools/bench_flat_bf16.py [--min-ms 150] [--arms fp32,workaround,bf16] [--out results.json]"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_bf16 import gpu_info  # noqa: E402

WORKLOAD = "flat7_620_b4"
ARMS = ("fp32", "workaround", "bf16")


class Arm:
    def __init__(self, step, z, target, cast):
        self.step, self.z, self.target, self.cast = step, z.detach().requires_grad_(True), target, cast
        self.one = torch.ones((), device=z.device)
        self.graph = None

    def run(self):
        out = self.step(self.z.float() if self.cast else self.z, self.target)
        return out, torch.autograd.grad(out.loss, self.z, grad_outputs=self.one)[0]

    def capture(self):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                self.run()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.keep = self.run()  # the graph's outputs live as long as the graph
        torch.cuda.synchronize()


def check(arm16, arm_up):
    """bf16 step == fp32 step on the upcast logits: confusion and ratios bit-exact, scalars to 1e-5, dlogits within one
    bf16 rounding (2^-8 relative) plus 1e-5 of the largest gradient."""
    out, g = arm16.run()
    ref, g_ref = arm_up.run()
    torch.cuda.synchronize()
    a, r = g.double(), g_ref.double()
    grad_ok = bool(((a - r).abs() <= 2.0 ** -8 * r.abs() + 1e-5 * r.abs().max() + 1e-12).all())
    s, sr = out.scalars.double(), ref.scalars.double()
    scal_ok = bool(((s - sr).abs() <= 1e-5 * sr.abs() + 1e-5 * sr.abs().max()).all())
    return {"confusion_equal": bool(torch.equal(out.confusion[0], ref.confusion[0])),
            "ratios_equal": bool(torch.equal(out.ratios[0], ref.ratios[0])), "scalars_close": scal_ok,
            "dlogits_bf16": g.dtype == torch.bfloat16, "dlogits_close": grad_ok}


def peak_mb(arm):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    res = arm.run()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    del res
    return round(peak / 1e6, 1)


def launches(arm):
    from torch.profiler import ProfilerActivity, profile
    arm.run()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        arm.run()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return {"count": len(names), "kernels": sorted(n.split("(")[0] for n in names)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-ms", type=float, default=150.0, help="timed work per arm (ms)")
    ap.add_argument("--arms", default=",".join(ARMS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_flat_bf16 measures on a CUDA device; none is visible")
    import bench
    import rhseg_b200 as rh
    from rhseg_b200 import native
    arms_wanted = args.arms.split(",")
    wl = bench.WORKLOADS[WORKLOAD]
    dev = torch.device("cuda:0")
    data = bench.synth_inputs(wl, wl["B"], seed=1000, device=dev)
    z32, target = data["host"]["logits"], data["host"]["target"]
    z16 = z32.to(torch.bfloat16)
    step = rh.FusedFlatStep(wl["K"], data["weights"][0])
    make = {"fp32": lambda: Arm(step, z32, target, False), "workaround": lambda: Arm(step, z16, target, True),
            "bf16": lambda: Arm(step, z16, target, False)}
    res = {"gpu": gpu_info(), "workload": WORKLOAD, "library": native.LIB_PATH, "batch": wl["B"]}
    if "bf16" in arms_wanted:
        res["check"] = check(make["bf16"](), Arm(step, z16.float(), target, False))
    arms = {k: make[k]() for k in arms_wanted}
    res["peak_mb"] = {k: peak_mb(a) for k, a in arms.items()}
    for a in arms.values():
        a.capture()
        for _ in range(5):
            a.graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    first = next(iter(arms.values()))
    e0.record()
    first.graph.replay()
    e1.record()
    torch.cuda.synchronize()
    reps = max(5, int(25.0 / max(e0.elapsed_time(e1), 1e-3)))  # about 25 ms of replays per block
    times = {k: [] for k in arms}
    timed = {k: 0.0 for k in arms}
    while min(timed.values()) < args.min_ms or min(len(v) for v in times.values()) < 8:
        for k, a in arms.items():
            e0.record()
            for _ in range(reps):
                a.graph.replay()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            timed[k] += ms
            times[k].append(ms / reps)
    res["ms_per_step"] = {k: round(statistics.median(v), 4) for k, v in times.items()}
    res["timing"] = {"blocks": {k: len(v) for k, v in times.items()}, "steps_per_block": reps,
                     "timed_ms": {k: round(v, 1) for k, v in timed.items()},
                     "spread_ms": {k: [round(min(v), 4), round(max(v), 4)] for k, v in times.items()}}
    for a in arms.values():
        a.graph = a.keep = None
    res["launches_per_step"] = {k: launches(a) for k, a in arms.items()}
    line = json.dumps(res)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
