"""Validation pass of the hierarchical model (the reference's test(), train.py:324-339): five routes per workload and
feature dtype, one JSON line.

  dropin    the drop-in modules the way test() calls them: the head under no_grad, CE + Dice per level, the consistency
            term, and the five metric wrappers per level on the composed probabilities, eager
  step      FusedHierStep under no_grad (the training-path evaluation: other numbers, for scale), eager
  step_graph  the same, replayed from a CUDA graph
  validate  FusedHierStep.validate, eager
  graph     FusedHierStep.validate replayed from a CUDA graph

For each workload, in a process of its own: bench.synth_inputs (seed 1000, as tools/bench_bf16.py), per dtype (fp32,
bf16) the peak allocated memory of one call per route above what the inputs hold, kernel launches per call
(torch.profiler), the median of alternating timed blocks (>= --min-ms of work per route), and the per-kernel device time
of the validation and evaluation kernels with the bytes each must move (computed from the shapes) and the fraction of
the data sheet's 7.7 TB/s HBM bandwidth that this implies.
--fuse-eval root|all selects which levels of upsampled heads validate evaluates inside the band forward (the last level
always is; default: the package's default).
    python tools/bench_validate.py [--workloads a,b] [--dtypes fp32,bf16] [--fuse-eval root|all] [--out results.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_bf16 import gpu_info  # noqa: E402

WORKLOADS = ["unet_tl_620_b4", "hrnet_w48_tl_620_b4", "hrnet_w48_ext_620_b4"]
ROUTES = ["dropin", "step", "step_graph", "validate", "graph"]
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}
HBM_BYTES_PER_S = 7.7e12


def make_routes(rh, wl, data, feats, dev):
    from rhseg_b200.Metrics import losses, performance_metrics as pm
    tree = rh.ClassTree(wl["tree"])
    h = data["host"]
    params = [[p.to(dev) for p in h[k]] for k in ("hw", "hb", "fw", "fb")]
    target = h["target"].to(dev)
    out_size = None if wl["scale"] == 1 else (wl["H"], wl["W"])
    step = rh.FusedHierStep(tree, data["weights"])
    chans = tree.head_channels
    ch_off = [sum(chans[:L]) for L in range(len(chans))]
    tgt = [target[:, o:o + k] for o, k in zip(ch_off, chans)]
    ce, dice = losses.CrossEntropyLoss(), losses.SoftDiceLoss()
    mets = [pm.DiceScore(), pm.Jaccardindex(), pm.Accuracy(), pm.Precision(), pm.Recall()]

    def dropin():
        with torch.no_grad():
            probs, logits = rh.hier_head_forward(tree, feats, *params, out_size)
            loss = 0.0
            for L in range(len(chans)):
                loss = loss + ce(logits[L], tgt[L], True, data["weights"][L])
                d = dice(logits[L], tgt[L], True, data["weights"][L])
                loss = loss + (d if d is not None else 0.0)
            loss = loss + losses.hierarchical_consistency_loss(probs, tree.levels, tree.parent_of)
            metrics = [[m(probs[L], tgt[L], dev, chans[L], L != 0) for m in mets] for L in range(len(chans))]
        return loss, metrics

    def train_no_grad():
        with torch.no_grad():
            return step(feats, *params, target, out_size)

    def validate():
        return step.validate(feats, *params, target, out_size)

    graphs = {}

    def capture():
        for key, fn in (("step_graph", train_no_grad), ("graph", validate)):
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    fn()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                keep = fn()  # the graph's outputs live as long as the graph
            torch.cuda.synchronize()
            graphs[key] = (g, keep)

    return {"dropin": dropin, "step": train_no_grad, "step_graph": lambda: graphs["step_graph"][0].replay(),
            "validate": validate, "graph": lambda: graphs["graph"][0].replay()}, capture


def peak_mb(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    r = fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    del r
    return round(peak / 2 ** 20, 1)


def profile(fn):
    from torch.profiler import ProfilerActivity, profile as prof_
    fn()
    torch.cuda.synchronize()
    with prof_(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                  key=lambda e: e.time_range.start)


def level_bytes(wl, tree, B):
    """bytes each level's evaluation kernel must move: rhseg_level_eval_composed (logits, probabilities and targets,
    plus the parents' probability planes) and rhseg_level_eval (logits and targets, plus the parents' target planes and
    the previous level's index map, and its own index map unless it is the last level)"""
    N = wl["H"] * wl["W"]
    n = tree.num_levels
    val, ev = [], []
    for L, K in enumerate(tree.head_channels):
        G = tree.group_count(L) if L > 0 else 0
        val.append(B * N * 4 * (3 * K + G))
        ev.append(B * N * (4 * (2 * K + G) + (1 if L > 0 else 0) + (1 if L < n - 1 else 0)))
    return val, ev


def kernel_rates(events, name, bytes_per_level, levels):
    out = []
    ks = [e for e in events if name + "<" in e.name]
    for e, L in zip(ks, levels):
        us = e.device_time_total
        out.append({"level": L, "us": round(us, 1), "MB": round(bytes_per_level[L] / 1e6, 1),
                    "hbm_fraction": round(bytes_per_level[L] / (us * 1e-6) / HBM_BYTES_PER_S, 3)})
    return out


def one_dtype(rh, wl, data, dname, args, dev):
    feats = [f.to(DTYPES[dname]).contiguous() for f in data["host"]["feats"]]
    routes, capture = make_routes(rh, wl, data, feats, dev)
    res = {"peak_mb": {r: peak_mb(routes[r]) for r in ("dropin", "step", "validate")}}
    capture()
    tree = rh.ClassTree(wl["tree"])
    n = tree.num_levels
    ev = {r: profile(routes[r]) for r in ROUTES}
    res["launches_per_call"] = {r: len(v) for r, v in ev.items()}
    val_b, ev_b = level_bytes(wl, tree, wl["B"])
    eval_levels = list(range(n)) if wl["scale"] == 1 else list(range(1, n - 1))  # the rest: fused into the band forward
    from rhseg_b200 import head
    val_levels = list(range(n)) if wl["scale"] == 1 else ([] if head._FUSE_EVAL_VAL == "all" else list(range(1, n - 1)))
    res["kernels"] = {"level_val_pipe_kernel": kernel_rates(ev["validate"], "level_val_pipe_kernel", val_b, val_levels),
                      "level_eval_pipe_kernel": kernel_rates(ev["step"], "level_eval_pipe_kernel", ev_b, eval_levels)}
    for fn in routes.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {r: [] for r in ROUTES}
    timed = {r: 0.0 for r in ROUTES}
    while min(timed.values()) < args.min_ms or min(len(v) for v in times.values()) < 8:
        for r in ROUTES:
            reps = 3 if r == "dropin" else 10
            e0.record()
            for _ in range(reps):
                routes[r]()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            timed[r] += ms
            times[r].append(ms / reps)
    res["ms_per_call"] = {r: round(statistics.median(v), 4) for r, v in times.items()}
    res["spread_ms"] = {r: [round(min(v), 4), round(max(v), 4)] for r, v in times.items()}
    del routes
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return res


def one_workload(name, args):
    import rhseg_b200 as rh
    from rhseg_b200 import head
    import bench
    if args.fuse_eval:
        head._FUSE_EVAL_VAL = args.fuse_eval
    wl = bench.WORKLOADS[name]
    dev = torch.device("cuda:0")
    data = bench.synth_inputs(wl, wl["B"], seed=1000, device=dev)
    res = {"workload": name, "batch": wl["B"], "fuse_eval": head._FUSE_EVAL_VAL}
    for d in args.dtypes.split(","):
        res[d] = one_dtype(rh, wl, data, d, args, dev)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--dtypes", default="fp32,bf16")
    ap.add_argument("--one", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--min-ms", type=float, default=150.0, help="timed work per route, dtype and workload (ms)")
    ap.add_argument("--fuse-eval", default=None, choices=["root", "all"])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.one:
        print(json.dumps(one_workload(args.one, args)))
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench_validate measures on a CUDA device; none is visible")
    res = {"gpu": gpu_info(), "workloads": []}
    for name in args.workloads.split(","):
        cmd = [sys.executable, os.path.abspath(__file__), "--one", name, "--min-ms", str(args.min_ms), "--dtypes", args.dtypes]
        if args.fuse_eval:
            cmd += ["--fuse-eval", args.fuse_eval]
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
