"""The donor backbones, the flat -> hierarchy stitching and ProcessClasses against what the unmodified reference computes
for the same seeded inputs, stored in tests/golden/reference_pins.npz (tests/golden/make_reference_golden.py).  Where
the reference tree is present (oracle/ref_loader.py) they are also compared with the reference itself; the module
drop-in check imports the reference's train.py and runs only there."""
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader  # noqa: E402

REF = ref_loader.reference_root()
needs_reference = pytest.mark.skipif(not ref_loader.available(), reason="reference tree not present")
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_reference_golden as G  # noqa: E402
from helpers import close  # noqa: E402

PINS = np.load(G.PINS, allow_pickle=False)


def _ref():
    import ref_shim
    return ref_shim, ref_shim.load_reference()


def _check_backbone(rec, prefix):
    """A record of make_reference_golden against the stored one: identical key lists, outputs within 1e-5."""
    for k in [k for k in PINS.files if k.startswith(prefix + ".") and k.endswith("keys")]:
        assert json.loads(rec[k]) == json.loads(str(PINS[k])), k
    for out in sorted({k.rsplit(".", 1)[0] for k in PINS.files if k.startswith(prefix + ".") and k.endswith(".sample")}):
        assert list(rec[out + ".shape"]) == list(PINS[out + ".shape"]), out
        assert np.array_equal(rec[out + ".index"], PINS[out + ".index"]), out
        close(torch.from_numpy(rec[out + ".sample"]), torch.from_numpy(PINS[out + ".sample"]), what=out + " sample")
        close(torch.from_numpy(rec[out + ".channel_sums"]), torch.from_numpy(PINS[out + ".channel_sums"]), what=out + " channel sums")


def test_unet_donor_matches_reference_backbone():
    from rhseg_b200.Models import models
    tree = G.trees()["ext"]
    ours = G.unet_record(models, tree)
    _check_backbone(ours, "unet")
    assert json.loads(ours["unet.tables"]) == json.loads(str(PINS["unet.tables"]))
    if ref_loader.available():  # the reference itself, same parameters and input: bit for bit
        _, (rmodels, _, _) = _ref()
        theirs = G.unet_record(rmodels, tree)
        assert ours["unet.keys"] == theirs["unet.keys"] and ours["unet.tables"] == theirs["unet.tables"]
        assert np.array_equal(ours["unet.out.sample"], theirs["unet.out.sample"])
        assert np.array_equal(ours["unet.out.channel_sums"], theirs["unet.out.channel_sums"])


def test_hrnet_donor_matches_reference_backbone():
    from rhseg_b200.Models import models
    tree = G.trees()["tl"]
    ours = G.hrnet_record(models, tree, G.hrnet_config())
    assert list(ours["hrnet.out.shape"]) == [1, 720, 16, 24]
    _check_backbone(ours, "hrnet")
    if ref_loader.available():  # the reference's own config and modules
        ref_shim, (rmodels, _, _) = _ref()
        theirs = G.hrnet_record(rmodels, tree, ref_shim.hrnet_config())
        _check_backbone(theirs, "hrnet")
        assert ours["hrnet.keys"] == theirs["hrnet.keys"] and ours["hrnet.flat_keys"] == theirs["hrnet.flat_keys"]


@needs_reference
def test_module_dropin_shadows_reference_modules():
    """INTEGRATION.md section 1: with the package directory ahead of the reference root, the reference's
    train.py imports OUR Models / Metrics / tree_util."""
    import subprocess
    code = r"""
import sys
sys.path.insert(0, %r); import ref_shim
for n in ("timm","timm.models","timm.models.vision_transformer","segmentation_models_pytorch","torchmetrics","yacs","yacs.config",
          "matplotlib","matplotlib.pyplot","skimage","skimage.io","skimage.transform"):
    ref_shim._stub(n)
sys.modules["yacs.config"].CfgNode = ref_shim.CfgNode
sys.path[:0] = [%r, %r, %r]
import train
pkg = %r
assert train.models.__file__.startswith(pkg), train.models.__file__
assert train.losses.__file__.startswith(pkg), train.losses.__file__
assert train.performance_metrics.__file__.startswith(pkg)
import tree_util; assert tree_util.__file__.startswith(pkg)
import Data.dataset as d; assert d.__file__.startswith(%r)
fns = [[train.losses.CrossEntropyLoss(), train.losses.SoftDiceLoss(num_classes=4)]]
print("ok")
""" % (os.path.join(ROOT, "tests", "golden"), ROOT, os.path.join(ROOT, "restrictive-hierarchical-semantic-segmentation_b200"), REF,
       os.path.join(ROOT, "restrictive-hierarchical-semantic-segmentation_b200"), REF)
    env = dict(os.environ)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=REF, env=env, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_oracle_stitching_matches_reference_predicteval():
    """oracle.stitch_flat_to_levels == predictEval.get_parent_masks + combine_levels on both shipped trees."""
    from oracle import hier_oracle as O
    ours = G.stitch_record(lambda flat, tgt, tree: O.stitch_flat_to_levels(flat, tree))
    want = {k: PINS[k] for k in PINS.files if k.startswith("stitch.")}
    assert sorted(ours) == sorted(want) and all(np.array_equal(ours[k], want[k]) for k in want)
    if ref_loader.available():
        _ref()
        theirs = G.stitch_record(G.reference_stitch())
        assert sorted(theirs) == sorted(want) and all(np.array_equal(theirs[k], want[k]) for k in want)


def test_oracle_process_classes_pinned_to_reference():
    """ProcessClasses (Metrics/performance_metrics.py:27-47) is torch-only: the reference's own class pins the oracle's
    restatement (and through it the CUDA confusion kernels) on the three kinds of input that reach it (SURVEY.md 3.4):
    masked one-hots, composed probabilities, ties / all-zero pixels."""
    from oracle import hier_oracle as O
    ours = G.process_classes_record(O.process_classes)
    want = {k: PINS[k] for k in PINS.files if k.startswith("process_classes.")}
    assert sorted(ours) == sorted(want) and all(np.array_equal(ours[k], want[k]) for k in want)
    if ref_loader.available():
        _ref()
        theirs = G.process_classes_record(ref_loader.load_reference_module("Metrics.performance_metrics").ProcessClasses())
        assert all(np.array_equal(theirs[k], want[k]) for k in want)
