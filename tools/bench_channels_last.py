"""Channels-last donor features through the fused training step (FusedHierStep): three routes per workload and dtype,
one JSON line.

  nchw    contiguous features (the step as it has always run)
  copy    channels-last features through the old route: an explicit .contiguous() before the step and a
          .contiguous(memory_format=torch.channels_last) on dfeats (what a channels-last donor paid before the NHWC kernels)
  native  channels-last features read in place (RHSEG_FEATS_NHWC), dfeats written channels-last

For each workload, in a process of its own: bench.synth_inputs (seed 1000, as tools/bench_bf16.py), per dtype (fp32,
bf16) a check of the native route against the nchw route at the timed size, the peak allocated memory of one eager
step per route (above what the inputs hold), every route captured in a CUDA graph, warmed up and timed in alternating
blocks of graph replays (>= --min-ms of timed work per route), reported as the median block; with --kernels the
per-kernel device time of one eager step of the nchw and native routes (torch.profiler, after timing).
    python tools/bench_channels_last.py [--workloads a,b] [--dtypes fp32,bf16] [--kernels] [--out results.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_bf16 import WORKLOADS, Step, gpu_info, kernel_table  # noqa: E402

CL = torch.channels_last
ROUTES = ["nchw", "copy", "native"]
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}


class CopyStep(Step):
    """channels-last leaves, made contiguous for the step; dfeats converted back to channels-last"""

    def run(self):
        n = len(self.feats)
        out = self.fused([f.contiguous() for f in self.feats], *self.params, self.target, self.out_size)
        grads = torch.autograd.grad(out.loss, self.leaves, grad_outputs=self.one)
        return out, tuple(g.contiguous(memory_format=CL) for g in grads[:n]) + tuple(grads[n:])


def make(route, rh, wl, data, feats, dev):
    if route == "nchw":
        return Step(rh, wl, data, [f.contiguous() for f in feats], dev)
    cl = [f.contiguous(memory_format=CL) for f in feats]
    return (CopyStep if route == "copy" else Step)(rh, wl, data, cl, dev)


def check(out, grads, ref, ref_grads, n, fullres):
    """native route against the nchw route"""
    def close(a, r, rtol=1e-5):
        a, r = a.detach().double(), r.detach().double()
        return bool(((a - r).abs() <= rtol * r.abs() + rtol * r.abs().max() + 1e-12).all())
    res = {"scalars": close(out.scalars, ref.scalars)}
    if fullres:  # bit-identical where both kernels get the same resident wave (same psum grouping): DESIGN.md 3.8
        res["logits_probs_confusion_equal"] = all(torch.equal(a, b) for a, b in zip(out.logits + out.probs + out.confusion,
                                                                                    ref.logits + ref.probs + ref.confusion))
    else:
        # low-res tiles split between two CTAs add their partial sums in another order (as tools/bench_bf16.py: 2e-5)
        res["logits_probs_2e-5"] = all(close(a, b, 2e-5) for a, b in zip(out.logits + out.probs, ref.logits + ref.probs))
    res["dfeats_channels_last"] = all(g.is_contiguous(memory_format=CL) and not g.is_contiguous() for g in grads[:n])
    res["dfeats_last_level_equal"] = bool(torch.equal(grads[n - 1], ref_grads[n - 1])) if fullres else None
    tol = 2.0 ** -7 if grads[0].dtype == torch.bfloat16 else 1e-5
    res["dfeats_close"] = all(close(a, b, tol) for a, b in zip(grads[:n], ref_grads[:n]))
    res["params_1e-5"] = all(close(a, b) for a, b in zip(grads[n:], ref_grads[n:]))
    res["all_ok"] = all(v for v in res.values() if v is not None)
    return res


def peak_mb(step):
    """peak allocated memory of one eager step (forward + backward, outputs and gradients held) above the inputs"""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out, grads = step.run()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    del out, grads
    return round(peak / 2 ** 20, 1)


def one_dtype(rh, bench, wl, data, dname, args, dev):
    feats = [f.to(DTYPES[dname]) for f in data["host"]["feats"]]
    n = len(feats)
    fullres = wl["scale"] == 1
    steps = {r: make(r, rh, wl, data, feats, dev) for r in ROUTES}
    out, grads = steps["native"].run()
    ref, ref_grads = steps["nchw"].run()
    torch.cuda.synchronize()
    res = {"check": check(out, grads, ref, ref_grads, n, fullres)}
    del out, grads, ref, ref_grads
    res["peak_mb"] = {r: peak_mb(steps[r]) for r in ROUTES}
    for st in steps.values():
        st.capture()
    for st in steps.values():
        for _ in range(5):
            st.graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    steps["nchw"].graph.replay()
    e1.record()
    torch.cuda.synchronize()
    reps = max(5, int(25.0 / max(e0.elapsed_time(e1), 1e-3)))
    times = {r: [] for r in ROUTES}
    timed = {r: 0.0 for r in ROUTES}
    while min(timed.values()) < args.min_ms or min(len(v) for v in times.values()) < 8:
        for r, st in steps.items():
            e0.record()
            for _ in range(reps):
                st.graph.replay()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            timed[r] += ms
            times[r].append(ms / reps)
    ms = {r: statistics.median(v) for r, v in times.items()}
    res["ms_per_step"] = {r: round(v, 4) for r, v in ms.items()}
    res["native_vs_nchw"] = round(ms["native"] / ms["nchw"], 3)
    res["native_vs_copy"] = round(ms["native"] / ms["copy"], 3)
    res["timing"] = {"blocks": len(times["nchw"]), "steps_per_block": reps,
                     "spread_ms": {r: [round(min(v), 4), round(max(v), 4)] for r, v in times.items()}}
    for st in steps.values():
        st.graph = None
        st.keep = None
    if args.kernels:
        res["kernels_us"] = {r: kernel_table(steps[r]) for r in ("nchw", "native")}
    del steps
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return res


def one_workload(name, args):
    import rhseg_b200 as rh
    import bench
    wl = bench.WORKLOADS[name]
    dev = torch.device("cuda:0")
    data = bench.synth_inputs(wl, wl["B"], seed=1000, device=dev)
    res = {"workload": name, "batch": wl["B"]}
    for d in args.dtypes.split(","):
        res[d] = one_dtype(rh, bench, wl, data, d, args, dev)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--dtypes", default="fp32,bf16")
    ap.add_argument("--one", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--min-ms", type=float, default=150.0, help="timed work per route, dtype and workload (ms)")
    ap.add_argument("--kernels", action="store_true", help="per-kernel device time of one eager step (nchw, native)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.one:
        print(json.dumps(one_workload(args.one, args)))
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench_channels_last measures on a CUDA device; none is visible")
    res = {"gpu": gpu_info(), "workloads": []}
    for name in args.workloads.split(","):
        cmd = [sys.executable, os.path.abspath(__file__), "--one", name, "--min-ms", str(args.min_ms), "--dtypes", args.dtypes]
        if args.kernels:
            cmd.append("--kernels")
        r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
        if r.returncode != 0:
            res["workloads"].append({"workload": name, "error": r.stderr[-2000:]})
            continue
        res["workloads"].append(json.loads(r.stdout.strip().splitlines()[-1]))
    line = json.dumps(res)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
