"""Generates tests/golden/reference_pins.npz: what tests/test_reference_gated.py compares the donor backbones, the flat ->
hierarchy stitching and ProcessClasses against, stored so that those comparisons run without the reference tree.

    python tests/golden/make_reference_golden.py                 # from the reference's own modules (needs the tree)
    python tests/golden/make_reference_golden.py --source pinned # from this repository's implementations

With the reference tree present (see oracle/ref_loader.py) every record comes from the reference: Models.models UNet /
HighResolutionNet, predictEval.combine_levels, Metrics.performance_metrics.ProcessClasses.  The committed file was made
with --source pinned: from the donors of Models/models.py, oracle.stitch_flat_to_levels and oracle.process_classes of
the commit whose tests/test_reference_gated.py held each of them equal to the reference on these same inputs (exactly
for UNet, stitching and ProcessClasses; within 1e-5 for HRNet).  `source` in the file says which.

Donor parameters are not the reference's random init (a UNet state dict is 54 MB): every tensor of the state dict is
drawn by name from a seeded generator, so both implementations get identical parameters from their key lists alone.
Backbone outputs are stored as per-channel sums plus a seeded sample of elements."""
import argparse
import json
import os
import sys
import zlib

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import hier_oracle as O  # noqa: E402
from oracle import ref_loader  # noqa: E402

PINS = os.path.join(HERE, "reference_pins.npz")
N_SAMPLE = 4096


def _stage(n, branches, block, blocks, channels):
    return {"NUM_MODULES": n, "NUM_BRANCHES": branches, "BLOCK": block, "NUM_BLOCKS": blocks, "NUM_CHANNELS": channels,
            "FUSE_METHOD": "SUM"}


# HRNetV2-W48: the MODEL.* entries of the reference's config that HighResolutionNet reads (65.9 M parameters with the
# hierarchical head of class_tree_tl.json)
HRNET_W48 = {"ALIGN_CORNERS": True, "EXTRA": {
    "FINAL_CONV_KERNEL": 1,
    "STAGE1": _stage(1, 1, "BOTTLENECK", [4], [64]),
    "STAGE2": _stage(1, 2, "BASIC", [4, 4], [48, 96]),
    "STAGE3": _stage(4, 3, "BASIC", [4, 4, 4], [48, 96, 192]),
    "STAGE4": _stage(3, 4, "BASIC", [4, 4, 4, 4], [48, 96, 192, 384])}}


def hrnet_config():
    return ref_loader.CfgNode({"MODEL": HRNET_W48})


def trees():
    """class_tree_tl.json and class_tree_tl_extended.json, as recorded in the head fixtures made from them."""
    return {name: json.loads(str(np.load(os.path.join(HERE, fx + ".npz"))["tree"]))
            for name, fx in (("tl", "unet_tl"), ("ext", "unet_ext"))}


def seed_parameters(model, seed=0):
    """Every floating tensor of the state dict drawn from a generator seeded by its name (fan-in scaled weights, norm
    weights near 1, positive running variances); integer buffers are left alone."""
    with torch.no_grad():
        for name, t in model.state_dict().items():
            if not t.is_floating_point():
                continue
            g = torch.Generator().manual_seed(seed ^ zlib.crc32(name.encode()))
            r = torch.randn(t.shape, generator=g)
            if name.endswith("running_var"):
                v = 0.75 + 0.25 * r.tanh()
            elif name.endswith("running_mean") or (t.dim() == 1 and name.endswith("bias")):
                v = 0.1 * r
            elif t.dim() == 1:
                v = 1.0 + 0.1 * r
            else:
                v = r / (t.numel() / t.shape[0]) ** 0.5
            t.copy_(v)


def _keys(model):
    return json.dumps([[k, list(v.shape)] for k, v in model.state_dict().items()])


def _summary(prefix, y):
    """Per-channel sums (fp64) and N_SAMPLE elements at seeded distinct positions of a backbone output."""
    y = y.detach()
    g = torch.Generator().manual_seed(zlib.crc32(prefix.encode()))
    idx = torch.randperm(y.numel(), generator=g)[:N_SAMPLE].sort().values
    return {prefix + ".shape": np.asarray(y.shape), prefix + ".channel_sums": y.double().sum(dim=[0] + list(range(2, y.dim()))).numpy(),
            prefix + ".index": idx.numpy(), prefix + ".sample": y.reshape(-1)[idx].numpy()}


def unet_record(models, tree):
    torch.manual_seed(0)
    m = models.UNet(size=64, n_channels=3, hierarchy=tree, model_type=1).eval()
    seed_parameters(m)
    x = torch.randn(2, 3, 40, 56, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        y = m._run_unet(x)
    rec = {"unet.keys": _keys(m), "unet.tables": json.dumps([m.levels, m.parent_of, m.child_groups, m.children_of])}
    rec.update(_summary("unet.out", y))
    return rec


def hrnet_record(models, tree, cfg):
    torch.manual_seed(0)
    m = models.HighResolutionNet(cfg, hierarchy=tree, model_type=1).eval()
    seed_parameters(m)
    x = torch.randn(1, 3, 64, 96, generator=torch.Generator().manual_seed(2))
    with torch.no_grad():
        y = m._forward_backbone(x)
    flat = models.HighResolutionNet(cfg, hierarchy=tree, model_type=0).eval()
    seed_parameters(flat)
    with torch.no_grad():
        z = flat(x)[1]
    rec = {"hrnet.keys": _keys(m), "hrnet.flat_keys": _keys(flat)}
    rec.update(_summary("hrnet.out", y))
    rec.update(_summary("hrnet.flat_out", z))
    return rec


def stitch_inputs(trees_):
    """The seeded flat predictions of the stitching test, per tree: (flat one-hots, flat targets)."""
    g = torch.Generator().manual_seed(3)
    out = {}
    for name, tree in trees_.items():
        n = sum(1 for lv in O.hierarchy_tables(tree)[0] for c in lv if not _children(tree, c))
        lab = torch.randint(0, n, (2, 9, 11), generator=g)
        flat = torch.nn.functional.one_hot(lab, n).permute(0, 3, 1, 2).float()
        tgt = torch.nn.functional.one_hot(torch.randint(0, n, (2, 9, 11), generator=g), n).permute(0, 3, 1, 2).float()
        out[name] = (flat, tgt)
    return out


def _children(tree, name):
    stack = [tree]
    while stack:
        d = stack.pop()
        if name in d:
            return d[name]
        stack.extend(v for v in d.values() if isinstance(v, dict))
    return {}


def process_classes_inputs():
    """The seeded inputs of the ProcessClasses test: (K, prediction kind, p, tgt) with kind 0 = masked one-hots,
    1 = probabilities with all-zero pixels and exact ties."""
    g = torch.Generator().manual_seed(9)
    out = []
    for K in (1, 2, 3, 4, 7):
        B, H, W = 2, 13, 17
        lab = torch.randint(0, K, (B, H, W), generator=g)
        onehot = torch.nn.functional.one_hot(lab, K).permute(0, 3, 1, 2).float()
        ignore = torch.rand(B, 1, H, W, generator=g) < 0.3
        masked = torch.where(ignore, torch.zeros_like(onehot), onehot)            # train.py:230
        probs = torch.rand(B, K, H, W, generator=g)
        probs[:, :, :2] = 0.0                                                     # nothing positive
        probs[:, :, 2:4] = probs[:, :1, 2:4]                                      # exact ties
        tgt = torch.nn.functional.one_hot(torch.randint(0, K, (B, H, W), generator=g), K).permute(0, 3, 1, 2).float()
        tgt = torch.where(torch.rand(B, 1, H, W, generator=g) < 0.4, torch.zeros_like(tgt), tgt)
        out += [(K, 0, masked, tgt), (K, 1, probs, tgt)]
    return out


def stitch_record(stitch):
    """stitch(flat, targets, tree) -> list of per-level tensors."""
    rec = {}
    for name, (flat, tgt) in stitch_inputs(trees()).items():
        for L, t in enumerate(stitch(flat, tgt, trees()[name])):
            rec["stitch.%s.%d" % (name, L)] = t.double().numpy()
    return rec


def process_classes_record(process_classes):
    """process_classes(p, tgt, child) -> (predictions, targets)."""
    rec = {}
    for K, kind, p, tgt in process_classes_inputs():
        for child in (False, True):
            a, b = process_classes(p, tgt, child)
            key = "process_classes.%d.%d.%d" % (K, kind, int(child))
            rec[key + ".pred"], rec[key + ".target"] = a.double().numpy(), b.double().numpy()
    return rec


def reference_stitch():
    """predictEval.get_parent_masks + combine_levels, called the way the reference's evaluation calls them."""
    import importlib
    for n in ("matplotlib.colors", "skimage.measure", "skimage.color", "scipy", "sklearn"):
        ref_loader._stub(n)
    pe = importlib.import_module("predictEval")

    def stitch(flat, tgt, tree):
        names = [n for n in pe.bfs_order(tree) if not pe.children_map(tree).get(n)]
        par, _, _ = pe.get_parent_masks([flat], [tgt], tree, {n: i for i, n in enumerate(names)})
        parent_order = [n for n in pe.bfs_order(tree) if pe.children_map(tree).get(n)]
        return pe.combine_levels([flat], par, tree, names, parent_order)
    return stitch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--source", choices=["reference", "pinned"], default="reference")
    args = ap.parse_args()
    tr = trees()
    if args.source == "reference":
        models, _, _ = ref_loader.load_reference()
        stitch = reference_stitch()
        process_classes = ref_loader.load_reference_module("Metrics.performance_metrics").ProcessClasses()
    else:
        import rhseg_b200  # noqa: F401
        from rhseg_b200.Models import models
        stitch, process_classes = (lambda flat, tgt, tree: O.stitch_flat_to_levels(flat, tree)), O.process_classes
    rec = {"source": np.asarray(args.source), "trees": np.asarray(json.dumps(tr)), "hrnet_config": np.asarray(json.dumps(HRNET_W48))}
    rec.update(unet_record(models, tr["ext"]))
    rec.update(hrnet_record(models, tr["tl"], hrnet_config()))
    rec.update(stitch_record(stitch))
    rec.update(process_classes_record(process_classes))
    rec = {k: (np.asarray(v) if isinstance(v, str) else v) for k, v in rec.items()}
    np.savez_compressed(PINS, **rec)
    print("wrote", PINS, "(%d bytes, source %s)" % (os.path.getsize(PINS), args.source))


if __name__ == "__main__":
    main()
