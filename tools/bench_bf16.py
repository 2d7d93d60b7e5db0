"""fp32 vs bf16 donor features through the fused training step (FusedHierStep), one JSON line.

For each workload, in a process of its own: bench.synth_inputs (seed 1000, drawn on the GPU as bench.py does for its
extra configurations), a check that the bf16 step equals the fp32 step on the upcast features (the bounds of
tests/test_gpu_bf16_features.py), both steps captured in CUDA graphs, warmed up, then timed in alternating blocks of
graph replays (>= --min-ms of timed work per dtype) and reported as the median block.  Also: Mpixel/s, the bf16
algorithmic bytes (bench.py's formulas with 2-byte feature elements) over the step time as a fraction of the
measured HBM bandwidth, the conv backward alone (20 back-to-back launches between one CUDA event pair) in both
dtypes and, with --kernels, the per-kernel device time of one eager step of each dtype (torch.profiler, after timing).
    python tools/bench_bf16.py [--workloads a,b] [--kernels] [--out results.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = ["hrnet_w48_tl_620_b4", "unet_tl_620_b4", "hrnet_w48_ext_620_b4", "unet_tl_1024_b8"]
BF_FEAT = 2  # bytes per bf16 feature element


def bf16_bytes(bench, wl, B):
    """bench.algorithmic_bytes with the feature reads (forward, backward) and the dfeats write at 2 bytes."""
    alg = bench.algorithmic_bytes(wl, B)
    _, _, chans, _ = bench.tree_shape(wl)
    h, w = bench.feat_hw(wl)
    feat32 = B * wl["C"] * h * w * 4  # one level's feature tensor in fp32
    saved = len(chans) * 3 * feat32 * (4 - BF_FEAT) // 4  # forward read + backward read + dfeats write, per level
    conv_bwd = [b - 2 * feat32 * (4 - BF_FEAT) // 4 for b in alg["conv_bwd"]]  # backward read + dfeats write
    return dict(step=alg["step"] - saved, step_fp32=alg["step"], conv_bwd=conv_bwd, conv_bwd_fp32=alg["conv_bwd"])


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else ""
    f = [x.strip() for x in line.split(",")]
    return {"name": f[0], "power_limit": f[1], "sm_clock_max": f[2]} if len(f) == 3 else {"raw": line}


class Step:
    """One fused step (forward + backward to every leaf) on fixed buffers, capturable."""

    def __init__(self, rh, wl, data, feats, dev):
        self.fused = rh.FusedHierStep(rh.ClassTree(wl["tree"]), data["weights"])
        h = data["host"]
        self.feats = [f.detach().requires_grad_(True) for f in feats]
        self.params = [[p.to(dev).requires_grad_(True) for p in h[k]] for k in ("hw", "hb", "fw", "fb")]
        self.target = h["target"].to(dev)
        self.out_size = None if wl["scale"] == 1 else (wl["H"], wl["W"])
        self.leaves = self.feats + [p for grp in self.params for p in grp]
        self.one = torch.ones((), device=dev)
        self.graph = None

    def run(self):
        out = self.fused(self.feats, *self.params, self.target, self.out_size)
        grads = torch.autograd.grad(out.loss, self.leaves, grad_outputs=self.one)
        return out, grads

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


def check_equal(out, grads, ref, ref_grads, n_feats):
    """bf16 step == fp32 step on the upcast features, within the bounds of tests/test_gpu_bf16_features.py."""
    def close(a, r, rtol):
        a, r = a.detach().double(), r.detach().double()
        return bool(((a - r).abs() <= rtol * r.abs() + rtol * r.abs().max() + 1e-12).all())
    res = {"scalars": close(out.scalars, ref.scalars, 1e-5),
           "logits": all(close(a, b, 2e-5) for a, b in zip(out.logits, ref.logits)),
           "probs": all(close(a, b, 2e-5) for a, b in zip(out.probs, ref.probs)),
           "params": all(close(a, b, 1e-5) for a, b in zip(grads[n_feats:], ref_grads[n_feats:]))}
    ok_d = True
    for a, r in zip(grads[:n_feats], ref_grads[:n_feats]):
        a, r = a.double(), r.double()
        ok_d &= bool(((a - r).abs() <= 2.0 ** -8 * r.abs() + 1e-5 * r.abs().max()).all())
    res["dfeats"] = ok_d and all(g.dtype == torch.bfloat16 for g in grads[:n_feats])
    conf = []
    for a, b, z in zip(out.confusion, ref.confusion, ref.logits):
        top = z.topk(2, dim=1).values if z.shape[1] > 1 else None
        margin = (top[:, 0] - top[:, 1]).min().item() if top is not None else float("inf")
        conf.append(bool(torch.equal(a, b)) if margin >= 1e-5 else None)
    res["confusion_equal_where_margin_ge_1e-5"] = conf
    res["all_ok"] = all(v for k, v in res.items() if k != "confusion_equal_where_margin_ge_1e-5") and all(c is not False for c in conf)
    return res


def conv_bwd_alone(native, wl, B, feats_L, K, reps=20):
    h, w = bench_mod.feat_hw(wl)
    dev = feats_L.device
    dz = torch.randn(B, K, h, w, device=dev)
    eff = torch.randn(B, K, wl["C"], device=dev)
    df = torch.empty_like(feats_L)
    S = torch.zeros(B, K, wl["C"], dtype=torch.float64, device=dev)
    s = torch.zeros(B, K, dtype=torch.float64, device=dev)
    flag = native.FEATS_BF16 if feats_L.dtype == torch.bfloat16 else 0
    cur = torch.cuda.current_stream().cuda_stream

    def run():
        native.call("rhseg_head_conv_bwd", feats_L.data_ptr(), dz.data_ptr(), eff.data_ptr(), B, wl["C"], K, h * w,
                    df.data_ptr(), S.data_ptr(), s.data_ptr(), flag, cur)
    for _ in range(2):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_table(step):
    from torch.profiler import ProfilerActivity, profile
    step.run()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step.run()
        torch.cuda.synchronize()
    tot = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            k = e.name.split("(")[0][:120]
            tot[k] = tot.get(k, 0.0) + e.device_time_total
    return {k: round(v, 1) for k, v in sorted(tot.items(), key=lambda kv: -kv[1])}


def one_workload(name, args):
    import rhseg_b200 as rh
    from rhseg_b200 import native
    global bench_mod
    import bench as bench_mod
    wl = bench_mod.WORKLOADS[name]
    B = wl["B"]
    dev = torch.device("cuda:0")
    data = bench_mod.synth_inputs(wl, B, seed=1000, device=dev)
    feats32 = data["host"]["feats"]
    feats16 = [f.to(torch.bfloat16) for f in feats32]
    n = len(feats32)
    # correctness at the timed size: bf16 step vs the fp32 step on the upcast features
    s16 = Step(rh, wl, data, feats16, dev)
    sup = Step(rh, wl, data, [f.float() for f in feats16], dev)
    out, grads = s16.run()
    ref, ref_grads = sup.run()
    torch.cuda.synchronize()
    check = check_equal(out, grads, ref, ref_grads, n)
    del out, grads, ref, ref_grads, sup
    torch.cuda.empty_cache()
    s32 = Step(rh, wl, data, feats32, dev)
    s32.capture()
    s16.capture()
    steps = {"fp32": s32, "bf16": s16}
    for st in steps.values():  # warm both graphs
        for _ in range(5):
            st.graph.replay()
    torch.cuda.synchronize()
    # block size: about 25 ms of replays per block
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    s32.graph.replay()
    e1.record()
    torch.cuda.synchronize()
    per = max(e0.elapsed_time(e1), 1e-3)
    reps = max(5, int(25.0 / per))
    times = {"fp32": [], "bf16": []}
    timed = {"fp32": 0.0, "bf16": 0.0}
    while min(timed.values()) < args.min_ms or min(len(v) for v in times.values()) < 8:
        for k, st in steps.items():
            e0.record()
            for _ in range(reps):
                st.graph.replay()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            timed[k] += ms
            times[k].append(ms / reps)
    ms = {k: statistics.median(v) for k, v in times.items()}
    peaks, peak_src = bench_mod.load_peaks()
    bb = bf16_bytes(bench_mod, wl, B)
    _, _, chans, _ = bench_mod.tree_shape(wl)
    dom = max(range(n), key=lambda L: bb["conv_bwd"][L])
    del steps, s32, s16
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    cb = {"level": dom, "K": chans[dom], "ms_bf16": conv_bwd_alone(native, wl, B, feats16[dom], chans[dom]),
          "ms_fp32": conv_bwd_alone(native, wl, B, feats32[dom], chans[dom])}
    cb["frac_hbm_bf16"] = bb["conv_bwd"][dom] / (cb["ms_bf16"] * 1e-3) / 1e9 / peaks["hbm_gbs"]
    cb["frac_hbm_fp32"] = bb["conv_bwd_fp32"][dom] / (cb["ms_fp32"] * 1e-3) / 1e9 / peaks["hbm_gbs"]
    px = B * wl["H"] * wl["W"]
    res = {"workload": name, "batch": B, "check": check,
           "ms_per_step": {k: round(v, 4) for k, v in ms.items()}, "speedup_bf16": round(ms["fp32"] / ms["bf16"], 3),
           "mpix_per_s": {k: round(px / (v * 1e-3) / 1e6, 1) for k, v in ms.items()},
           "alg_bytes_mb": {"bf16": round(bb["step"] / 1e6, 1), "fp32": round(bb["step_fp32"] / 1e6, 1)},
           "frac_hbm_bf16_step": round(bb["step"] / (ms["bf16"] * 1e-3) / 1e9 / peaks["hbm_gbs"], 3),
           "frac_hbm_fp32_step": round(bb["step_fp32"] / (ms["fp32"] * 1e-3) / 1e9 / peaks["hbm_gbs"], 3),
           "conv_bwd_alone": {k: (round(v, 4) if isinstance(v, float) else v) for k, v in cb.items()},
           "timing": {"blocks": {k: len(v) for k, v in times.items()}, "steps_per_block": reps,
                      "timed_ms": {k: round(v, 1) for k, v in timed.items()},
                      "spread_ms": {k: [round(min(v), 4), round(max(v), 4)] for k, v in times.items()}},
           "hbm_peak_gbs": peaks["hbm_gbs"], "hbm_peak_source": peak_src}
    if args.kernels:
        res["kernels_us"] = {}
        for k, fe in (("fp32", feats32), ("bf16", feats16)):
            res["kernels_us"][k] = kernel_table(Step(rh, wl, data, fe, dev))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--one", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--min-ms", type=float, default=150.0, help="timed work per dtype and workload (ms)")
    ap.add_argument("--kernels", action="store_true", help="per-kernel device time of one eager step per dtype")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.one:
        print(json.dumps(one_workload(args.one, args)))
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench_bf16 measures on a CUDA device; none is visible")
    res = {"gpu": gpu_info(), "workloads": []}
    for name in args.workloads.split(","):
        cmd = [sys.executable, os.path.abspath(__file__), "--one", name, "--min-ms", str(args.min_ms)]
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
