#!/usr/bin/env python
"""Benchmark of the restrictive-hierarchy head + loss + metrics path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

One "step" = the body of the reference's train_epoch (train.py:201-241) minus the donor backbone and the optimiser,
on synthetic per-level donor features:
    head forward (per-level feats -> probs, logits)  ->  train-path prediction + confusion-matrix metrics  ->
    CE + Dice per level + consistency  ->  backward to per-level dfeats and head / FiLM parameter gradients.
`value` is whole-job Mpixel/s (B*H*W pixels per step per GPU) with inputs resident in HBM; `e2e` is the same step
driven from pinned HOST buffers (H2D of the step's features and targets and D2H of the loss + metrics inside the timed
region).  The headline (`value`, `ms_per_step`) times exactly K steps, back to back, with a CUDA event between
consecutive steps, and reports the MEDIAN step; the secondary timings (`e2e`, `dropin_modules`, `roofline`) take their
own step counts, derived from K.  `configs` holds one short measurement of every other BASELINE.json configuration.

--dump-outputs DIR writes what the last timed step returned to its caller as DIR/<name>.npy (float32, or float64 for
the int64 confusion matrices and fp64 buffers): loss, scalars, per-level ratios / confusion / probs / logits, and the
gradients of every input.  Arrays too large to keep whole are stored as a fixed, seeded sample of their flattened
elements (files named *_sampled.npy), at most 64 MB in all.  Inputs are seeded, so two builds run with the same
arguments can be compared file for file.

Prints ONE JSON line on rank 0.  `--impl reference` times the reference's own modules (oracle/_ref: byte copies of
Models/, Metrics/, train.py staged by tools/stage_reference.py) on the host cores, same workload, same batch.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)

import torch  # noqa: E402

from tools import synth  # noqa: E402  (neutral input generator: neither product nor oracle)

TL = {"background": {}, "upper": {}, "lower": {}, "tooth": {"pulp": {}, "dentin": {}, "enamel": {}, "composite": {}}}
EXT = {"background": {}, "tooth+alveolar": {"alveolar": {"upper": {}, "lower": {}},
                                            "tooth": {"composite": {}, "healthy": {"pulp": {}, "dentin": {}, "enamel": {}}}}}
FLAT7 = {n: {} for n in ("background", "upper", "lower", "pulp", "dentin", "enamel", "composite")}  # leaves of TL
W_TL = [[0.0297, 1.577, 0.9619, 0.1770], [1.5432, 0.2638, 1.0413, 3.9722]]  # reference README.md:71
W_FLAT = [[0.0285, 1.5159, 0.9227, 1.4842, 0.2532, 1.0, 3.8021]]            # reference README.md:79

# BASELINE.json configs -> workloads.  B is the per-GPU batch (weak scaling) unless strong=True (B is the GLOBAL batch,
# split over the ranks).
WORKLOADS = {
    "hrnet_w48_tl_620_b4": dict(tree=TL, kind="hrnet", C=720, H=620, W=620, scale=4, B=4, weights=W_TL, cfg="configs[1]"),
    "unet_tl_620_b4": dict(tree=TL, kind="unet", C=64, H=620, W=620, scale=1, B=4, weights=W_TL, cfg="configs[0]"),
    "hrnet_w48_ext_620_b4": dict(tree=EXT, kind="hrnet", C=720, H=620, W=620, scale=4, B=4, weights=None, cfg="configs[2]"),
    "unet_ext_620_b4": dict(tree=EXT, kind="unet", C=64, H=620, W=620, scale=1, B=4, weights=None, cfg="configs[2] (UNet donor)"),
    "flat7_620_b4": dict(tree=FLAT7, kind="flat", K=7, C=0, H=620, W=620, scale=1, B=4, weights=W_FLAT, cfg="configs[3]"),
    "unet_tl_1024_b8": dict(tree=TL, kind="unet", C=64, H=1024, W=1024, scale=1, B=8, weights=W_TL, cfg="configs[4] per-GPU share at 8 GPUs"),
    "unet_tl_1024_b64": dict(tree=TL, kind="unet", C=64, H=1024, W=1024, scale=1, B=64, weights=W_TL, strong=True, cfg="configs[4]"),
}
DEFAULT_WORKLOAD = "hrnet_w48_tl_620_b4"
EXTRA_CONFIGS = ["unet_tl_620_b4", "hrnet_w48_ext_620_b4", "flat7_620_b4", "unet_tl_1024_b64"]
STEP_TEXT = {
    "hier": "head fwd + train-path prediction + 5 confusion metrics + CE/Dice/consistency + bwd (dfeats, head+FiLM grads)",
    "flat": "flat 7-class logits: train-path prediction + 5 confusion metrics + weighted CE/Dice + bwd (dlogits)",
}


def feat_hw(wl):
    if wl["scale"] == 1:
        return wl["H"], wl["W"]
    return (wl["H"] + wl["scale"] - 1) // wl["scale"], (wl["W"] + wl["scale"] - 1) // wl["scale"]


def local_batch(wl, world, rank=0):
    if not wl.get("strong"):
        return wl["B"]
    base, rem = divmod(wl["B"], world)
    return base + (1 if rank < rem else 0)


def tree_shape(wl):
    levels, groups = synth.tree_levels_groups(wl["tree"])
    chans = [len(lv) for lv in levels]
    return levels, groups, chans, [0] + [len(g) for g in groups]


def algorithmic_bytes(wl, B):
    """SURVEY.md 8(d) formulas, fp32, every API-visible tensor moved once per pass."""
    _, _, chans, gcount = tree_shape(wl)
    h, w = feat_hw(wl)
    N, Nf, C = wl["H"] * wl["W"], h * w, wl["C"]
    out = dict(fwd=0, loss=0, bwd=0, metrics=0, conv_bwd=[], fwd_conv=[])
    if wl["kind"] == "flat":  # loss fwd: read z,t; bwd: read z,t write dz; metrics: read z,t
        K = wl["K"]
        out["loss"] = B * (4 * K + 4 * K) * N
        out["bwd"] = B * (4 * K + 4 * K + 4 * K) * N
        out["metrics"] = B * (4 * K + 4 * K) * N
        out["dom"] = [B * (4 * K + 4 * K + 4 * K) * N]
    else:
        for K, g in zip(chans, gcount):
            out["fwd"] += B * (4 * C * Nf + 2 * 4 * K * N + 4 * g * N)
            out["loss"] += B * (4 * K + 4 * K) * N
            out["bwd"] += B * (2 * 4 * C * Nf + (4 * K + 4 * K + 4 * g) * N)
            out["metrics"] += B * (4 * K + 4 * K) * N
            # dominant kernel (1x1-conv backward): read feats + write dfeats + read dz at feature res
            out["conv_bwd"].append(B * (2 * 4 * C * Nf + 4 * K * Nf))
            out["fwd_conv"].append(B * (4 * C * Nf + 4 * K * Nf))
        out["dom"] = out["conv_bwd"]
    out["step"] = out["fwd"] + out["loss"] + out["bwd"]
    return out


def config_of(name, wl, world):
    """The `config` object: identical in both arms (ours / --impl reference) for the same command line."""
    _, _, chans, _ = tree_shape(wl)
    B = local_batch(wl, world)
    fbytes = len(chans) * B * wl["C"] * feat_hw(wl)[0] * feat_hw(wl)[1] * 4 if wl["kind"] != "flat" else B * wl["K"] * wl["H"] * wl["W"] * 4 * 2
    return {"workload": name, "baseline_config": wl["cfg"], "tree_levels": chans, "feat_channels": wl["C"],
            "batch_per_gpu": B, "global_batch": wl["B"] if wl.get("strong") else B * world,
            "image": [wl["H"], wl["W"]], "feat_hw": list(feat_hw(wl)),
            "step": STEP_TEXT["flat" if wl["kind"] == "flat" else "hier"],
            "l2_policy": "inputs larger than L2 (%.0f MB of inputs per step vs 126 MB L2)" % (fbytes / 1e6)}


def synth_inputs(wl, B, seed, device="cpu", pin=False, notooth_sample=None):
    """SURVEY.md 8(d) synthetic inputs: N(0,1) features per level, ternary targets built with the dataset's ignore
    rule, default-style head / FiLM parameter init.  device="cpu": host tensors (optionally pinned); a CUDA device:
    everything is drawn on the GPU (the extra configurations, whose host-side generation would take minutes)."""
    levels, groups, chans, _ = tree_shape(wl)
    h, w = feat_hw(wl)
    dev = torch.device(device)
    g = torch.Generator(device=dev).manual_seed(seed)
    C = wl["C"]
    host = {}
    if wl["kind"] == "flat":
        host["logits"] = torch.randn(B, wl["K"], wl["H"], wl["W"], generator=g, device=dev) * 2
        host["feats"], host["hw"], host["hb"], host["fw"], host["fb"] = [], [], [], [], []
    else:
        host["feats"] = [torch.randn(B, C, h, w, generator=g, device=dev) for _ in chans]
        bound = 1.0 / (C ** 0.5)
        host["hw"] = [(torch.rand(k, C, 1, 1, generator=g, device=dev) * 2 - 1) * bound for k in chans]
        host["hb"] = [(torch.rand(k, generator=g, device=dev) * 2 - 1) * bound for k in chans]
        host["fw"] = [(torch.rand(2 * C, kp, generator=g, device=dev) * 2 - 1) / (kp ** 0.5) for kp in chans[:-1]]
        host["fb"] = [(torch.rand(2 * C, generator=g, device=dev) * 2 - 1) / (kp ** 0.5) + 1.0 for kp in chans[:-1]]
    tl = synth.synth_targets(levels, groups, B, wl["H"], wl["W"], g, device=dev)
    if notooth_sample is not None and len(levels) > 1 and groups[0]:
        tl = synth.drop_class_in_sample(tl, levels, groups, notooth_sample, groups[0][0][0])
    host["target"] = torch.cat(tl, dim=1).contiguous()  # NCHW like the dataset's tensors (cat of one permuted one-hot keeps its layout)
    del tl
    weights = wl["weights"] or [[1.0] * k for k in chans]
    if pin:
        host["feats"] = [f.pin_memory() for f in host["feats"]]
        host["target"] = host["target"].pin_memory()
        if "logits" in host:
            host["logits"] = host["logits"].pin_memory()
    return dict(levels=levels, groups=groups, chans=chans, weights=weights, host=host)


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
class GpuStep:
    """Device-resident state + the step through the package's public API."""

    def __init__(self, wl, data, device):
        import rhseg_b200
        from rhseg_b200 import metric_ops
        from rhseg_b200.Metrics import losses
        self.rh, self.metric_ops, self.losses = rhseg_b200, metric_ops, losses
        self.wl, self.data, self.dev = wl, data, device
        self.flat = wl["kind"] == "flat"
        h = data["host"]
        self.target = h["target"].to(device)
        self.one = torch.ones((), device=device)  # d(loss)/d(loss), allocated once instead of a fill per step
        self.result = self.global_summary = self.maps = None
        self.keep_maps = False  # hold the step's probabilities and logits for --dump-outputs
        if self.flat:
            self.logits = h["logits"].to(device).requires_grad_(True)
            self.fused = rhseg_b200.FusedFlatStep(wl["K"], data["weights"][0])
            self.feats, self.params = [], [[], [], [], []]
            return
        self.tree = rhseg_b200.ClassTree(wl["tree"])
        self.feats = [f.to(device).requires_grad_(True) for f in h["feats"]]
        self.params = [[p.to(device).requires_grad_(True) for p in h[k]] for k in ("hw", "hb", "fw", "fb")]
        self.out_size = None if wl["scale"] == 1 else (wl["H"], wl["W"])
        self.ce, self.dice = losses.CrossEntropyLoss(), losses.SoftDiceLoss()
        self.fused = rhseg_b200.FusedHierStep(self.tree, data["weights"])
        # room behind the step summary for the head / FiLM parameter gradients (the data-parallel exchange buffer)
        self.fused.exchange_tail = sum(p.numel() for grp in self.params for p in grp)

    def input_bytes(self):
        if self.flat:
            return self.logits.numel() * 4 + self.target.numel() * 4
        return sum(f.numel() * 4 for f in self.feats) + self.target.numel() * 4

    def targets(self):
        out, s = [], 0
        for k in self.data["chans"]:  # channel slices of the wide target tensor (train.py:185-193)
            out.append(self.target[:, s:s + k])
            s += k
        return out

    def step(self):
        """Fused step (rhseg_b200.FusedHierStep / FusedFlatStep): the whole train_epoch body in one autograd node."""
        self.grads = self.maps = None  # free the previous step's gradient tensors first (they are GBs for the large batches)
        if self.flat:
            out = self.fused(self.logits, self.target)
            self.grads = torch.autograd.grad(out.loss, [self.logits], grad_outputs=self.one)
        else:
            hw, hb, fw, fb = self.params
            out = self.fused(self.feats, hw, hb, fw, fb, self.target, self.out_size)
            leaves = self.feats + [p for grp in self.params for p in grp]
            self.grads = torch.autograd.grad(out.loss, leaves, grad_outputs=self.one)  # dfeats per level + head / FiLM parameter grads
        self.result = (out.scalars, out.ratios)
        if self.keep_maps:  # not out.loss: it would keep the autograd graph of the step alive
            self.maps = (out.probs, out.logits)
        self.confusion, self.summary, self.exchange, self.global_summary = out.confusion, out.summary, out.exchange, out.global_summary
        return self.result

    def step_dropin(self):
        """Same work through the drop-in modules, called the way train.py calls them."""
        self.rh.clear_memo()
        hw, hb, fw, fb = self.params
        probs, logits = self.rh.hier_head_forward(self.tree, self.feats, hw, hb, fw, fb, self.out_size)
        targets = self.targets()
        onehots, ratios = [], []
        for L, z in enumerate(logits):  # train.py:206-232: prediction glue + the five metrics
            onehot, eval_t = self.metric_ops.predict_onehot(z.detach(), targets[L])
            ratios.append(self.metric_ops.level_ratios(onehot, eval_t, L != 0))
            onehots.append(onehot)
        loss = None
        for L, z in enumerate(logits):  # train.py:132-143
            w = self.data["weights"][L]
            ce = self.ce(z, targets[L], class_weight=w, logits_input=True)
            di = self.rh.level_loss(z, targets[L], w, 0.0, True).dice  # tensor form of SoftDiceLoss (no host sync)
            loss = ce + di if loss is None else loss + ce + di
        loss = loss + self.losses.hierarchical_consistency_loss(onehots, self.tree.levels, self.tree.parent_of)
        leaves = self.feats + [p for grp in self.params for p in grp]
        grads = torch.autograd.grad(loss, leaves)
        return loss.detach(), ratios, grads


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons = [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                sm.append(float(f[1]))
                out["sm_max_mhz"] = float(f[2])
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out["sm_mhz"] = statistics.median(sm)
        out["reasons"], out["samples"] = sorted(reasons), len(sm)
        return out


def kernels_per_call(name, upsampled):
    if name in ("rhseg_head_level_fwd", "rhseg_head_level_fwd_eval"):
        return 2 if upsampled else 1
    if name == "rhseg_head_conv_bwd_params":
        return 2
    return 1


class Harness:
    """One workload on this rank: state, the data-parallel exchange, CUDA-graph capture, block timing."""

    def __init__(self, args, name, rank, world, dev, pin_host):
        from rhseg_b200 import dist as rdist
        self.rdist = rdist
        self.args, self.name, self.rank, self.world, self.dev = args, name, rank, world, dev
        self.wl = wl = WORKLOADS[name]
        self.B = local_batch(wl, world, rank)
        # tens of GB per step (the 64-image batch on one or two GPUs): eager, a 20 ms step has no launch overhead to hide
        # and a captured graph would hold a second copy of every gradient tensor
        self.use_graph = bool(args.graph) and not (wl.get("strong") and world < 4)
        # the headline workload is generated on the host (its pinned buffers feed the end-to-end timing); the others on the GPU
        self.data = synth_inputs(wl, self.B, seed=1000 + rank, device="cpu" if pin_host else dev, pin=pin_host)
        self.st = GpuStep(wl, self.data, dev)
        self.px, self.kind = None, "none" if world == 1 else "nccl"
        self.graph = None
        if world > 1 and not self.st.flat:
            self._connect()

    # -- data-parallel exchange -----------------------------------------------------------------------------------
    def _connect(self):
        st, rdist = self.st, self.rdist
        st.step()  # sizes the exchange buffer
        torch.cuda.synchronize()
        if os.environ.get("RHSEG_EXCHANGE", "p2p") == "p2p":
            try:
                self.px = rdist.PeerExchange(st.exchange.numel())
                self.kind = "p2p"
            except Exception as e:
                sys.stderr.write("peer-memory exchange unavailable (%r); using NCCL\n" % (e,))
        if self.px is not None:
            reduce_fn = lambda s: self.px.all_reduce(s)  # noqa: E731  summary only: a few hundred bytes
        else:
            def reduce_fn(s):
                buf = s.clone()
                torch.distributed.all_reduce(buf)
                return buf
        # exact data-parallel gradients: the summary is summed over ranks between forward and backward
        st.fused.data_parallel(reduce_fn, self.world)

    def exchange(self):
        """The path's cross-rank traffic (pixel data never leaves its GPU): the step summary (loss terms, valid-sample
        counts, confusion matrices) is summed BETWEEN forward and backward inside the fused step (FusedHierStep.
        data_parallel); here, after the backward, ONE all-reduce of the head / FiLM parameter gradients (a few thousand
        floats).  Single node: one kernel over NVLink peer memory each (rhseg_xchg_all_reduce); RHSEG_EXCHANGE=nccl
        (or no P2P) -> rhseg_pack_f64 + NCCL."""
        st = self.st
        if self.world == 1 or st.flat:
            return
        grads = st.grads[len(st.feats):]
        n_sum = st.summary.numel()
        if self.px is not None:
            self.px.all_reduce(st.summary[:0], grads, out=st.exchange[n_sum:])
            return
        buf = self.rdist.pack_exchange(st.summary[:0], grads, out=None)
        torch.distributed.all_reduce(buf)
        st.exchange[n_sum:n_sum + buf.numel()].copy_(buf)

    def full_step(self):
        self.st.step()
        self.exchange()

    # -- timing ------------------------------------------------------------------------------------------------------
    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def capture(self):
        if not self.use_graph:
            return
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    self.full_step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.full_step()  # the exchanges are captured with the step (no host work per replay)
            g.replay()
            torch.cuda.synchronize()
            self.graph = g
        except Exception as e:  # capture is an optimisation, never a requirement
            sys.stderr.write("cuda graph capture unavailable (%r); timing eagerly\n" % (e,))
            self.graph = None
            torch.cuda.synchronize()

    def one_step(self):
        if self.graph is not None:
            self.graph.replay()
        else:
            self.full_step()

    def timed_steps(self, steps):
        """Exactly `steps` steps back to back between one barrier + synchronize on each side, a CUDA event on the
        launching stream before the first and after every step; max over ranks per step.  Returns the ms of every step."""
        self.barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record()
        for i in range(steps):
            self.one_step()
            ev[i + 1].record()
        self.barrier()
        t = torch.tensor([ev[i].elapsed_time(ev[i + 1]) for i in range(steps)], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return t.tolist()

    def close(self):
        self.graph = None
        if self.px is not None:
            self.px.check()  # raises if any exchange timed out (results would be NaN)
            self.px.close()
            self.px = None


def dp_check(args, rank, world, dev):
    """N > 1, once before timing: the batch-sharded step (one shard per rank, summary exchange between forward and
    backward, gradient exchange after) against the SAME global batch run as one single-process step on rank 0.
    Rank 1's first sample has no tooth (its deeper-level Dice is NaN: the valid-sample counts differ between ranks).
    Losses within 1e-5 relative, gradients within 1e-5 (relative to the tensor's largest entry), the exchanged confusion
    matrices equal to the exact integer sum of the ranks' matrices, and at most 1e-5 of the pixels moved against the
    single-process matrices (argmax near-ties, see below) -- or the run fails."""
    import rhseg_b200
    from rhseg_b200 import dist as rdist
    name = args.workload
    wl = WORKLOADS[name]
    if wl["kind"] == "flat":
        return None
    Bl = max(1, min(local_batch(wl, world, rank), 2))  # two samples per rank keep the global batch small
    Bg = Bl * world
    _, _, chans, _ = tree_shape(wl)
    # rank 0 draws the global batch on its GPU and broadcasts it; every rank keeps its shard
    data = synth_inputs(wl, Bg, seed=4242, device=dev, notooth_sample=Bl if world > 1 else None)
    h = data["host"]
    for t in h["feats"] + h["hw"] + h["hb"] + h["fw"] + h["fb"] + [h["target"]]:
        torch.distributed.broadcast(t, src=0)
    tree = rhseg_b200.ClassTree(wl["tree"])
    out_size = None if wl["scale"] == 1 else (wl["H"], wl["W"])
    sl = slice(rank * Bl, (rank + 1) * Bl)

    def leaves(s):
        return ([f[s].contiguous().requires_grad_(True) for f in h["feats"]],
                [[p.clone().requires_grad_(True) for p in h[k]] for k in ("hw", "hb", "fw", "fb")])

    # sharded
    step = rhseg_b200.FusedHierStep(tree, data["weights"])
    n_par = sum(p.numel() for k in ("hw", "hb", "fw", "fb") for p in h[k])
    step.exchange_tail = n_par
    px = None
    pf, pp = leaves(sl)
    probe = step(pf, *pp, h["target"][sl].contiguous(), out_size)
    if os.environ.get("RHSEG_EXCHANGE", "p2p") == "p2p":
        try:
            px = rdist.PeerExchange(probe.exchange.numel())
        except Exception:
            px = None
    if px is not None:
        step.data_parallel(lambda s: px.all_reduce(s), world)
    else:
        def nccl_sum(s):
            b = s.clone()
            torch.distributed.all_reduce(b)
            return b
        step.data_parallel(nccl_sum, world)
    feats, params = leaves(sl)
    out = step(feats, *params, h["target"][sl].contiguous(), out_size)
    flat_params = [p for grp in params for p in grp]
    grads = torch.autograd.grad(out.loss, feats + flat_params)
    pg = grads[len(feats):]
    if px is not None:
        red = px.all_reduce(out.summary[:0], pg)
    else:
        red = rdist.pack_exchange(out.summary[:0], pg)
        torch.distributed.all_reduce(red)
    conf_shapes = [tuple(c.shape) for c in out.confusion]
    glob = rdist.unpack_global(out.global_summary, len(chans), conf_shapes)
    xs = px.status() if px is not None else 0
    # single process on rank 0 (every rank computes it: simpler than shipping the gradients around, still one GPU each)
    ref_step = rhseg_b200.FusedHierStep(tree, data["weights"])
    rf, rp = leaves(slice(0, Bg))
    ro = ref_step(rf, *rp, h["target"], out_size)
    rflat = [p for grp in rp for p in grp]
    rg = torch.autograd.grad(ro.loss, rf + rflat)
    loss_rel = abs(glob["total"].item() - ro.loss.item()) / max(abs(ro.loss.item()), 1e-30)
    # integers: (1) the exchanged confusion matrices must equal the exact int64 sum over ranks of the local ones;
    # (2) against the single-process step a handful of pixels may move: its conv kernel splits the pixel tiles between
    # CTAs at other places (the split depends on the batch), logits differ in the last bit and exact near-ties of the
    # argmax flip -- reported as moved pixels, bounded at 1e-5 of the evaluated pixels
    conf_eq, moved = True, 0
    for L, (a, b) in enumerate(zip(glob["confusion"], ro.confusion)):
        local = out.confusion[L].clone()
        torch.distributed.all_reduce(local)
        conf_eq = conf_eq and torch.equal(a, local)
        moved += int((a - b).abs().sum().item()) // 2
    px_eval = Bg * wl["H"] * wl["W"] * len(chans)
    grad_rel, off = 0.0, 0
    for p, want in zip(flat_params, rg[len(rf):]):  # DDP mean over ranks of the parameter gradients
        got = (red[off:off + p.numel()] / world).view(want.shape)
        off += p.numel()
        grad_rel = max(grad_rel, ((got - want.double()).abs().max() / want.abs().max().clamp_min(1e-30)).item())
    for L in range(len(feats)):  # what the donor's DDP sees: local dfeats / world == the global step's dfeats of this shard
        want = rg[L][sl]
        grad_rel = max(grad_rel, ((grads[L] / world - want).abs().max() / want.abs().max().clamp_min(1e-30)).item())
    agg = torch.tensor([loss_rel, grad_rel, 0.0 if conf_eq else 1.0, float(xs), float(moved)], dtype=torch.float64, device=dev)
    torch.distributed.all_reduce(agg, op=torch.distributed.ReduceOp.MAX)
    if px is not None:
        px.close()
    n_valid = [int(glob["n_dice"][L].item()) for L in range(len(chans))]
    res = {"loss_rel": agg[0].item(), "confusion_equal": agg[2].item() == 0.0, "grad_rel": agg[1].item(),
           "xchg_status": int(agg[3].item()), "argmax_near_tie_pixels_moved_vs_single_process": int(agg[4].item()),
           "pixels_evaluated": px_eval, "global_batch": Bg, "dice_valid_samples_per_level": n_valid,
           "exchange": "p2p" if px is not None else "nccl",
           "what": "sharded (world=%d, %d samples per rank, rank 1 holds a sample without tooth) vs the same global batch in one process"
                   % (world, Bl)}
    del data, h, feats, params, rf, rp, rg, grads
    torch.cuda.empty_cache()
    if not (res["loss_rel"] <= 1e-5 and res["grad_rel"] <= 1e-5 and res["confusion_equal"] and res["xchg_status"] == 0
            and res["argmax_near_tie_pixels_moved_vs_single_process"] <= 1e-5 * px_eval):
        raise SystemExit("data-parallel check failed: %s" % json.dumps(res))
    return res


def measure_extra(args, name, rank, world, dev, peaks):
    """One of the other BASELINE.json configurations: same step, same block timing, short."""
    wl = WORKLOADS[name]
    hz = Harness(args, name, rank, world, dev, pin_host=False)
    for _ in range(3):
        hz.full_step()
    hz.capture()
    for _ in range(2):
        hz.one_step()
    torch.cuda.synchronize()
    big = wl.get("strong") and world < 4
    steps = 15 if big else 100
    times = hz.timed_steps(steps)
    ms = statistics.median(times)
    alg = algorithmic_bytes(wl, hz.B)
    px_total = sum(local_batch(wl, world, r) for r in range(world)) * wl["H"] * wl["W"]
    # dominant kernel, timed alone as back-to-back launches
    dom = dominant_alone(hz, alg)
    graph_used = hz.graph is not None
    hz.close()
    res = {"workload": name, "baseline_config": wl["cfg"], "scaling": "strong" if wl.get("strong") else "weak",
           "batch_per_gpu": hz.B, "ms_per_step": ms, "ms_per_step_min": min(times), "timed_steps": steps,
           "Mpx/s": px_total / (ms * 1e-3) / 1e6,
           "whole_step_frac": (alg["step"] + alg["metrics"]) / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
           "head_loss_fwd_bwd_frac": alg["step"] / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
           "dom_kernel": dom["kernel"], "dom_kernel_frac": dom["frac"](peaks["hbm_gbs"]), "dom_kernel_ms": dom["ms"],
           "cuda_graph": graph_used}
    hz.st = None
    del hz
    torch.cuda.empty_cache()
    return res


def dominant_alone(hz, alg):
    """The workload's dominant kernel as 20 back-to-back launches between one event pair (inputs far beyond L2)."""
    from rhseg_b200 import native
    st, wl, B, dev = hz.st, hz.wl, hz.B, hz.dev
    cur = torch.cuda.current_stream().cuda_stream
    if st.flat:
        def run():
            st.step()
        name, nbytes, reps = "flat step (level_eval + step_finalize + dz_fullres_fused)", alg["loss"] + alg["bwd"] + alg["metrics"], 20
    else:
        chans = hz.data["chans"]
        dom_l = max(range(len(chans)), key=lambda L: alg["conv_bwd"][L])
        K_dom, (hf, wf) = chans[dom_l], feat_hw(wl)
        iso = dict(dz=torch.randn(B, K_dom, hf, wf, device=dev), w=torch.randn(B, K_dom, wl["C"], device=dev),
                   df=torch.empty_like(st.feats[dom_l]), S=torch.zeros(B, K_dom, wl["C"], dtype=torch.float64, device=dev),
                   s=torch.zeros(B, K_dom, dtype=torch.float64, device=dev))

        def run():
            native.call("rhseg_head_conv_bwd", st.feats[dom_l].data_ptr(), iso["dz"].data_ptr(), iso["w"].data_ptr(), B, wl["C"], K_dom,
                        hf * wf, iso["df"].data_ptr(), iso["S"].data_ptr(), iso["s"].data_ptr(), 0, cur)
        name, nbytes = "conv_bwd_kernel (1x1-conv backward, level %d)" % dom_l, alg["conv_bwd"][dom_l]
        reps = 5 if B * wl["C"] * hf * wf * 4 > 4e9 else 20
    for _ in range(2):
        run()
    torch.cuda.synchronize()
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    i0.record()
    for _ in range(reps):
        run()
    i1.record()
    torch.cuda.synchronize()
    ms = i0.elapsed_time(i1) / reps
    return {"kernel": name, "ms": ms, "bytes": nbytes, "frac": lambda peak: nbytes / (ms * 1e-3) / 1e9 / peak}


def bind_to_gpu_numa(local_rank):
    """Pins this process (and with it the first-touch placement of its pinned host buffers) to the NUMA node its GPU
    hangs off, so that the end-to-end H2D copies do not cross the socket interconnect.  Best effort; returns what it did."""
    info = {"numa_node": None, "cpus": None}
    try:
        p = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        info["pci"] = bdf
        if node < 0:
            return info
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["numa_node"], info["cpus"] = node, len(allowed)
    except Exception as e:
        info["error"] = repr(e)[:80]
    return info


def gpu_topology():
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        return [l.rstrip() for l in out.splitlines() if l.strip() and not l.startswith(("Legend", "  "))][:12]
    except Exception:
        return None


def run_ours(args, rank, world, local_rank):
    from rhseg_b200 import native
    name = args.workload
    wl = WORKLOADS[name]
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    numa = bind_to_gpu_numa(local_rank) if world > 1 else None
    peaks, peak_src = load_peaks()
    check = dp_check(args, rank, world, dev) if (world > 1 and not args.no_dp_check) else None

    strong_big = wl.get("strong") and world < 4
    hz = Harness(args, name, rank, world, dev, pin_host=not strong_big)
    st, B = hz.st, hz.B
    st.keep_maps = bool(args.dump_outputs) and rank == 0
    upsampled = wl["scale"] != 1
    alg = algorithmic_bytes(wl, B)

    # kernel-launch accounting + live timing of the dominant kernel (1x1-conv backward)
    counted = {"n": 0}
    conv_events = []
    timing_on = {"v": False}
    raw_call = native.call

    def counting_call(cname, *a):
        # rhseg_head_conv_bwd_params: conv kernel + parameter-gradient kernel; a level without FiLM (film_w NULL) of a narrow
        # donor (B*C*K <= 4096) is ONE launch (include/rhseg_b200.h)
        counted["n"] += 1 if (cname == "rhseg_head_conv_bwd_params" and a[12] is None and a[3] * a[4] * a[5] <= 4096) else kernels_per_call(cname, upsampled)
        if timing_on["v"] and cname == "rhseg_head_conv_bwd_params":
            # the call launches the conv backward and the parameter-gradient kernel: issue the two launches it makes
            # separately (same kernels, same order, include/rhseg_b200.h) so that the event pair brackets the conv kernel only
            (feats, dz, eff_w, B_, C_, K_, n_pix, dfeats, S, s, flags, head_w, film_w, gb, psum, n_out, K_prev, d_hw, d_hb, d_fw,
             d_fb, g_prev, _ticket, stream) = a
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            raw_call("rhseg_head_conv_bwd", feats, dz, eff_w, B_, C_, K_, n_pix, dfeats, S, s, flags & 3, stream)
            e1.record()
            raw_call("rhseg_head_param_grads", S, s, head_w, film_w, gb, psum, n_out, B_, C_, K_, K_prev, d_hw, d_hb, d_fw, d_fb,
                     g_prev, 1 if (flags & 4) else 0, stream)
            conv_events.append((e0, e1))
        else:
            raw_call(cname, *a)

    import rhseg_b200.dist as dist_mod
    import rhseg_b200.fused as fused_mod
    import rhseg_b200.head as head_mod
    import rhseg_b200.loss_ops as loss_mod
    import rhseg_b200.metric_ops as met_mod
    for mod in (native, head_mod, loss_mod, met_mod, fused_mod):
        mod.call = counting_call
    del dist_mod

    # ---- device-resident timing (`value`) ----
    for _ in range(max(args.warmup, 3)):
        hz.full_step()
    hz.capture()
    for _ in range(3):
        hz.one_step()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    times = hz.timed_steps(args.steps)
    ms = statistics.median(times)
    dumped = collect_outputs(hz) if st.keep_maps else None
    st.keep_maps, st.maps = False, None
    counted["n"] = 0
    hz.full_step()  # one eager step: the launches of a step, counted
    launches_per_step = counted["n"]
    torch.cuda.synchronize()

    # ---- the same step through the drop-in modules (reference call sequence), eager ----
    dropin_ms = dropin_graph_ms = None
    if not args.no_dropin and not st.flat and not wl.get("strong"):
        for _ in range(3):
            st.step_dropin()
        torch.cuda.synchronize()
        reps = min(args.steps, 20)
        ts = []
        for _ in range(5):
            d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            d0.record()
            for _ in range(reps):
                st.step_dropin()
            d1.record()
            torch.cuda.synchronize()
            ts.append(d0.elapsed_time(d1) / reps)
        dropin_ms = statistics.median(ts)
        # the same call sequence replayed from a CUDA graph (what a caller gets who captures the loop body: no host work)
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                st.step_dropin()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            dg = torch.cuda.CUDAGraph()
            with torch.cuda.graph(dg):
                st.step_dropin()
            dg.replay()
            torch.cuda.synchronize()
            ts = []
            for _ in range(5):
                d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                d0.record()
                for _ in range(reps):
                    dg.replay()
                d1.record()
                torch.cuda.synchronize()
                ts.append(d0.elapsed_time(d1) / reps)
            dropin_graph_ms = statistics.median(ts)
            del dg
        except Exception as e:
            sys.stderr.write("drop-in route not capturable (%r)\n" % (e,))
            torch.cuda.synchronize()

    # ---- dominant-kernel timing, live, on the launching stream (eager steps, inputs > L2) ----
    nL = len(hz.data["chans"])
    conv_ms = None
    if not st.flat:
        timing_on["v"] = True
        for _ in range(min(args.steps, 20)):
            st.step()
        torch.cuda.synchronize()
        timing_on["v"] = False
        per_level = [[] for _ in range(nL)]
        for i, (a, b) in enumerate(conv_events):
            per_level[nL - 1 - (i % nL)].append(a.elapsed_time(b))  # backward visits the last level first
        conv_ms = [statistics.median(v) for v in per_level]
    alone = dominant_alone(hz, alg) if not args.no_alone else None
    clocks = sampler.stop() if rank == 0 else None

    # ---- end-to-end from pinned host buffers (`e2e`) ----
    e2e = None
    if not strong_big:
        e2e = time_e2e(args, hz)

    xchg_status = hz.px.status() if hz.px is not None else 0
    loss_value = float(st.result[0][0].item())
    graph_used = hz.graph is not None
    hz.close()
    if rank != 0:
        # the other ranks take part in the extra configurations' collectives
        if not args.no_configs and not args.workload_only:
            for extra in EXTRA_CONFIGS:
                if extra != name:
                    measure_extra(args, extra, rank, world, dev, peaks)
        return None

    px_total = sum(local_batch(wl, world, r) for r in range(world)) * wl["H"] * wl["W"]
    line = {
        "metric": "hier head+loss fwd+bwd Mpixel/s", "value": px_total / (ms * 1e-3) / 1e6, "unit": "Mpixel/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong" if wl.get("strong") else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config_of(name, wl, world),
        "timing": {"timed_steps": len(times), "ms_per_step_median": ms, "ms_per_step_min": min(times),
                   "ms_per_step_max": max(times), "timed_ms_total": sum(times),
                   "how": "barrier + synchronize, K steps (graph replays when captured) back to back with a CUDA event before the first and after each, barrier + synchronize; max over ranks per step; median step reported"},
        "run": {"api": "fused step (rhseg_b200.FusedHierStep)" if not st.flat else "fused flat step (rhseg_b200.FusedFlatStep)",
                "cuda_graph": graph_used, "loss": loss_value,
                "collective": ("summary all-reduce between fwd and bwd + head/FiLM gradient all-reduce after bwd, %s"
                               % {"p2p": "one peer-memory kernel over NVLink each (rhseg_xchg_all_reduce)", "nccl": "NCCL"}[hz.kind]) if world > 1 else "none",
                "xchg_status": xchg_status, "numa": numa, "topology": gpu_topology() if world > 1 else None},
        "step_bytes": {"algorithmic_head_loss_fwd_bwd": alg["step"], "metrics": alg["metrics"],
                       "frac_of_hbm_peak_head_loss_fwd_bwd": alg["step"] / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                       "frac_of_hbm_peak_whole_step": (alg["step"] + alg["metrics"]) / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                       "frac_of_nominal_8TBs_whole_step": (alg["step"] + alg["metrics"]) / (ms * 1e-3) / 1e9 / 8000.0},
        "clocks": clocks,
        "gpu_launches": launches_per_step * args.steps,
        "gpu_launches_per_step": launches_per_step,
    }
    if conv_ms is not None:
        dom = max(range(nL), key=lambda L: conv_ms[L])
        achieved = alg["conv_bwd"][dom] / (conv_ms[dom] * 1e-3) / 1e9
        line["roofline"] = {"kernel": "conv_bwd_kernel (1x1-conv backward, level %d)" % dom, "bound": "hbm", "achieved": achieved,
                            "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                            "traffic": load_traffic(name), "peak_source": peak_src,
                            "bytes_per_launch": alg["conv_bwd"][dom], "ms_per_launch": conv_ms[dom], "per_level_ms": conv_ms,
                            "timing": "in-step: one CUDA-event pair around each launch of the kernel inside eager steps (median; includes the launch gap the event pair itself opens)"}
    elif alone is not None:
        line["roofline"] = {"kernel": alone["kernel"], "bound": "hbm", "achieved": alone["bytes"] / (alone["ms"] * 1e-3) / 1e9,
                            "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": alone["frac"](peaks["hbm_gbs"]), "traffic": None,
                            "peak_source": peak_src, "bytes_per_launch": alone["bytes"], "ms_per_launch": alone["ms"]}
    if alone is not None and "roofline" in line and conv_ms is not None:
        line["roofline"]["alone"] = {"ms_per_launch": alone["ms"], "achieved": alone["bytes"] / (alone["ms"] * 1e-3) / 1e9,
                                     "frac": alone["frac"](peaks["hbm_gbs"]),
                                     "timing": "back-to-back launches of the same kernel between one event pair"}
    if e2e is not None:
        line["e2e"] = e2e
    if dropin_ms is not None:
        line["dropin_modules"] = {"ms_per_step": dropin_ms, "value": B * wl["H"] * wl["W"] / (dropin_ms * 1e-3) / 1e6, "unit": "Mpixel/s",
                                  "cuda_graph_ms_per_step": dropin_graph_ms,
                                  "cuda_graph_value": (B * wl["H"] * wl["W"] / (dropin_graph_ms * 1e-3) / 1e6) if dropin_graph_ms else None,
                                  "note": "same step through Models/Metrics drop-in modules in the reference's call order, this rank: eager (host-bound: ~40 launches + autograd + allocator per step) and the same calls replayed from a CUDA graph"}
    if check is not None:
        line["dp_check"] = check
    if not args.no_configs and not args.workload_only:
        line["configs"] = [{"workload": name, "baseline_config": wl["cfg"], "scaling": line["scaling"], "batch_per_gpu": B,
                            "ms_per_step": ms, "Mpx/s": line["value"],
                            "whole_step_frac": line["step_bytes"]["frac_of_hbm_peak_whole_step"],
                            "head_loss_fwd_bwd_frac": line["step_bytes"]["frac_of_hbm_peak_head_loss_fwd_bwd"],
                            "dom_kernel": line.get("roofline", {}).get("kernel"),
                            "dom_kernel_frac": alone["frac"](peaks["hbm_gbs"]) if alone else None}]
        for extra in EXTRA_CONFIGS:
            if extra != name:
                line["configs"].append(measure_extra(args, extra, rank, world, dev, peaks))
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_reference(name, wl, B, steps=3, warmup=1)  # ~20-30 s of host work
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    return line


def time_e2e(args, hz):
    """The same step driven from pinned HOST buffers: every step copies its features + targets host -> device (the copy
    of step i+1 overlaps step i on a copy stream) and reads loss + metrics back to the host."""
    st, data, dev, world = hz.st, hz.data, hz.dev, hz.world
    host = data["host"]
    flat = st.flat
    src_feats = [host["logits"]] if flat else host["feats"]
    # the ternary targets travel as int8 (the values the dataset produces: 1, 0, -1) and are widened on the device by
    # rhseg_targets_i8_to_f32 inside the step: a quarter of their fp32 bytes over PCIe
    tgt_host = host["target"].to(torch.int8).pin_memory()
    h2d = sum(f.numel() * 4 for f in src_feats) + tgt_host.numel()
    nres = 6 if flat else 2 + 4 * len(data["chans"])
    out_host = torch.empty(nres + sum(5 * (k + (1 if L else 0)) for L, k in enumerate(data["chans"])), dtype=torch.float32).pin_memory()
    d2h = out_host.numel() * 4
    cur_feats = [st.logits] if flat else st.feats
    # two device-side input sets: the H2D copy of step i+1 runs on a copy stream while step i computes
    target_f32 = st.target
    sets = [(cur_feats, torch.empty(st.target.shape, dtype=torch.int8, device=dev)),
            ([torch.empty_like(f).requires_grad_(True) for f in cur_feats], torch.empty(st.target.shape, dtype=torch.int8, device=dev))]
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def upload(i):
        feats_i, target_i = sets[i % 2]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i % 2])  # the step that last read this set has finished
            with torch.no_grad():
                for dst, src in zip(feats_i, src_feats):
                    dst.copy_(src, non_blocking=True)
                target_i.copy_(tgt_host, non_blocking=True)
            ready[i % 2].record(copy_stream)

    def e2e_step(i):
        upload(i + 1)                                   # prefetch the next step's inputs
        torch.cuda.current_stream().wait_event(ready[i % 2])
        if flat:
            st.logits, st.target = sets[i % 2][0][0], sets[i % 2][1]
        else:
            st.feats, st.target = sets[i % 2]
        scal, ratios = st.step()
        consumed[i % 2].record()
        hz.exchange()
        out_host.copy_(torch.cat([scal] + [r.flatten() for r in ratios]), non_blocking=True)
        torch.cuda.current_stream().synchronize()       # the caller reads loss / metrics on the host every step

    for ev in consumed:
        ev.record()
    upload(0)
    for i in range(2):
        e2e_step(i)
    e2e_steps = max(3, min(args.steps, 30))
    blocks, own, i = [], [], 2
    for _ in range(3):
        hz.barrier()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(e2e_steps):
            e2e_step(i)
            i += 1
        t1.record()
        hz.barrier()
        copy_stream.synchronize()
        t = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device=dev)
        own.append(t.item() / e2e_steps)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        blocks.append(t.item() / e2e_steps)
    if flat:
        st.logits, st.target = sets[0][0][0], target_f32
    else:
        st.feats, st.target = sets[0][0], target_f32
    e2e_ms = statistics.median(blocks)
    per_rank = [statistics.median(own)]
    if world > 1:
        allr = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        torch.distributed.all_gather(allr, torch.tensor([per_rank[0]], dtype=torch.float64, device=dev))
        per_rank = [t.item() for t in allr]
    px_total = sum(local_batch(hz.wl, world, r) for r in range(world)) * hz.wl["H"] * hz.wl["W"]
    return {"value": px_total / (e2e_ms * 1e-3) / 1e6, "unit": "Mpixel/s", "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "steps": e2e_steps, "blocks": len(blocks),
            "h2d_GBps_per_gpu": h2d / (e2e_ms * 1e-3) / 1e9,
            "h2d_GBps_per_rank": [h2d / (m * 1e-3) / 1e9 for m in per_rank],
            "note": "features (fp32) + ternary targets (int8, widened on the device) copied from pinned host memory every step "
                    "(copy of step i+1 overlaps step i); PCIe-bound"}


DUMP_BYTES = 64 << 20


def collect_outputs(hz):
    """Host copies of what the last step returned to its caller, name -> tensor (float32, or float64 for int64 and fp64
    results).  Arrays beyond a fair share of DUMP_BYTES keep a sample of their flattened elements at fixed, seeded
    positions: the same positions in every run with the same arguments."""
    st = hz.st
    scalars, ratios = st.result
    arrays = {"loss": scalars[:1], "scalars": scalars}  # StepOutput.loss is scalars[0]
    for L in range(len(ratios)):
        arrays["ratios_L%d" % L] = ratios[L]
        arrays["confusion_L%d" % L] = st.confusion[L]
    if st.flat:
        arrays["grad_logits"] = st.grads[0]
    else:
        for L in range(len(ratios)):
            arrays["probs_L%d" % L] = st.maps[0][L]
            arrays["logits_L%d" % L] = st.maps[1][L]
            arrays["grad_feats_L%d" % L] = st.grads[L]
        names = ["grad_%s_%d" % (key, i) for key, grp in zip(("head_w", "head_b", "film_w", "film_b"), st.params)
                 for i in range(len(grp))]
        arrays.update(zip(names, st.grads[len(st.feats):]))
        if hz.world > 1:
            arrays["exchange"] = st.exchange  # the step summary and the parameter gradients summed over the ranks
    large = [k for k, t in arrays.items() if t.numel() > 65536]
    small_bytes = sum(t.numel() * 8 for k, t in arrays.items() if k not in large)
    share = (DUMP_BYTES - small_bytes) // max(len(large), 1)  # bytes per large array
    res = {}
    for k, t in arrays.items():
        t = t.detach()
        wide = t.dtype in (torch.float64, torch.int64, torch.int32)
        n = share // (8 if wide else 4)
        if k in large and t.numel() > n:
            # n seeded draws, duplicates removed: distinct positions in increasing order (a permutation of all the
            # positions would take GBs of host memory for the largest outputs)
            g = torch.Generator().manual_seed(zlib.crc32(k.encode()))
            idx = torch.unique(torch.randint(0, t.numel(), (n,), generator=g))
            t, k = t.reshape(-1)[idx.to(t.device)], k + "_sampled"
        res[k] = t.to(torch.float64 if wide else torch.float32).cpu()
    return res


def write_outputs(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for k, t in arrays.items():
        np.save(os.path.join(path, k + ".npy"), t.numpy())


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "MEASURED_PEAKS.json (measured copy bandwidth on this pool's B200)"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback 6.65 TB/s (B200_PROFILING.md)"


def load_traffic(workload):
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(workload)
    except Exception:
        return None


# ------------------------------------------------------------------------------------------
# reference arm: the reference's own modules on the host cores (oracle/_ref), else the oracle port
# ------------------------------------------------------------------------------------------
def cpu_reference(name, wl, B, steps, warmup):
    from oracle import ref_bench
    torch.set_num_threads(os.cpu_count() or 1)
    data = synth_inputs(wl, B, seed=7, device="cpu")
    px = B * wl["H"] * wl["W"]
    _, _, chans, _ = tree_shape(wl)
    if ref_bench.available():
        sec, ts, loss = ref_bench.time_reference(wl, data, steps, warmup)
        kind = "reference"
        what = ("the reference's own Models.models / Metrics.losses / Metrics.performance_metrics / train.get_loss / "
                "train.get_metrics (byte copies under oracle/_ref; torchmetrics replaced by a restated stand-in), donor "
                "features patched in, loss.backward()")
    else:
        sec, ts, loss = port_reference(wl, data, steps, warmup)
        kind = "port"
        what = "oracle port of the reference CPU path (oracle/_ref not staged on this box)"
    return {"value": px / sec / 1e6, "unit": "Mpixel/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": "the full workload batch (%d images %dx%d, %d level(s)) per step, %d timed steps after %d warm-up, torch %s CPU fp32; %s"
                      % (B, wl["H"], wl["W"], len(chans), steps, warmup, torch.__version__, what),
            "ms_per_step": sec * 1e3, "ms_per_step_min": min(ts) * 1e3, "loss": loss}


def port_reference(wl, data, steps, warmup):
    from oracle import hier_oracle as O
    h = data["host"]
    levels, groups = data["levels"], data["groups"]
    _, parent_of, _, ogroups = O.hierarchy_tables(wl["tree"])
    out_size = None if wl["scale"] == 1 else (wl["H"], wl["W"])
    flat = wl["kind"] == "flat"
    leaves = [[t.clone().requires_grad_(True) for t in h[k]] for k in ("feats", "hw", "hb", "fw", "fb")]
    zflat = h["logits"].clone().requires_grad_(True) if flat else None
    targets, s = [], 0
    for k in data["chans"]:
        targets.append(h["target"][:, s:s + k])
        s += k

    def step():
        for grp in leaves:
            for t in grp:
                t.grad = None
        if flat:
            zflat.grad = None
            logits = [zflat]
        else:
            _, logits = O.head_forward(*leaves, levels, ogroups, out_size)
        onehots, eval_t = O.predict_onehot_masked([z.detach() for z in logits], targets)
        O.all_level_metrics(onehots, eval_t)
        loss, _ = O.total_loss(logits, targets, data["weights"], None if flat else onehots, levels, parent_of)
        loss.backward()
        return loss.item()

    loss = None
    for _ in range(warmup):
        loss = step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        loss = step()
        ts.append(time.perf_counter() - t0)
    return statistics.mean(ts), ts, loss


def run_reference(args, rank, world):
    if rank != 0:
        return None
    name = args.workload
    wl = WORKLOADS[name]
    B = local_batch(wl, world)
    if wl.get("strong") and B > 8:
        B = 8  # bounded sample of the 64-image batch (per-pixel normalised)
    base = cpu_reference(name, wl, B, steps=args.steps, warmup=args.warmup)
    return {"impl": "reference", "metric": "hier head+loss fwd+bwd Mpixel/s", "value": base["value"], "unit": "Mpixel/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["ms_per_step"],
            "higher_is_better": True, "scaling": "strong" if wl.get("strong") else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config_of(name, wl, world),
            "run": {"note": "rank 0's host cores only; value = pixels of ONE rank's batch / step time (the reference trains single-process)"},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the headline measurement (>= 1)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--graph", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-dropin", action="store_true", help="skip timing the drop-in module path (profiling runs)")
    ap.add_argument("--no-alone", action="store_true", help="skip the back-to-back timing of the dominant kernel (profiling runs)")
    ap.add_argument("--no-configs", action="store_true", help="skip the short measurement of the other BASELINE.json configurations")
    ap.add_argument("--workload-only", action="store_true", help="alias of --no-configs")
    ap.add_argument("--no-dp-check", action="store_true", help="N > 1: skip the sharded-vs-global-batch check before timing")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        line = run_reference(args, rank, world)
        if line is not None:
            print(json.dumps(line), flush=True)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    if world > 1:
        torch.cuda.set_device(local_rank)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        line = run_ours(args, rank, world, local_rank)
        if line is not None:
            print(json.dumps(line), flush=True)
    finally:
        if world > 1:
            torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
