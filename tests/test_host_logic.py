"""CPU-only checks: the C-ABI library loads and exports every symbol the header declares, the
compiled class-tree tables agree with the oracle's name-keyed structures, the product never
imports the oracle, the bench's byte model matches SURVEY.md 8(d), and the batch-sharded summary
exchange reproduces the single-process numbers (world_size-2 gloo)."""
import ast
import json
import os
import re
import socket
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "restrictive-hierarchical-semantic-segmentation_b200")

from oracle import hier_oracle as O  # noqa: E402

TL = {"background": {}, "upper": {}, "lower": {}, "tooth": {"pulp": {}, "dentin": {}, "enamel": {}, "composite": {}}}
EXT = {"background": {}, "tooth+alveolar": {"alveolar": {"upper": {}, "lower": {}},
                                            "tooth": {"composite": {}, "healthy": {"pulp": {}, "dentin": {}, "enamel": {}}}}}
ADV = {"a": {}, "b": {"b0": {}, "b1": {"b1x": {}}}, "c": {"c0": {}, "c1": {}, "c2": {}}}


def test_library_exports_every_declared_symbol():
    import rhseg_b200
    from rhseg_b200 import native
    header = open(os.path.join(ROOT, "include", "rhseg_b200.h")).read()
    declared = set(re.findall(r"\b(rhseg_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 20
    lib = native.lib()
    for name in sorted(declared):
        assert hasattr(lib, name), "library does not export %s" % name
    assert declared == set(native.SIGNATURES), (declared ^ set(native.SIGNATURES))
    assert lib.rhseg_abi_version() == 1
    assert b"invalid argument" in lib.rhseg_status_string(-1)


def test_argument_errors_do_not_need_a_gpu():
    from rhseg_b200 import native
    lib = native.lib()
    assert lib.rhseg_film_fold(None, None, None, None, None, 1.0, 1, 1, 1, 0, None, None, None, None) == -1
    assert lib.rhseg_loss_stats(None, None, 0, 0, 1, 4, 16, 1, None, None) == -1
    assert lib.rhseg_confusion_matrix(None, 0, 0, None, 0, 0, 1, 4, 16, 0, None, None) == -1
    with pytest.raises(native.NativeError):
        native.require_cuda(torch.zeros(2))
    with pytest.raises(native.NativeError):
        native.compile_level_table([0, 1, 0], 2)  # children of one parent must be contiguous


@pytest.mark.parametrize("tree", [TL, EXT, ADV, {"only": {}}, {"r": {"x": {"y": {"z": {}}}}}])
def test_tree_tables_match_oracle(tree):
    import rhseg_b200
    t = rhseg_b200.ClassTree(tree)
    levels, parent_of, children_of, groups = O.hierarchy_tables(tree)
    assert t.levels == levels and t.parent_of == parent_of and t.children_of == children_of
    assert t.child_groups == groups
    assert rhseg_b200.build_hierarchy_indices(tree) == (levels, parent_of, children_of)
    assert rhseg_b200.get_level_classes(tree, inc_parent=False) == O.names_per_depth(tree, parents_too=False)
    from rhseg_b200 import native
    M = native.MAX_K
    for L, tab in enumerate(t.host_tables):
        K = len(levels[L])
        assert tab[0] == K and tab[2] == (len(levels[L - 1]) if L else 0)
        if L == 0:
            assert tab[3] == native.ACT_SIGMOID and tab[4:4 + K] == [-1] * K
            continue
        assert tab[1] == len(groups[L - 1]) and tab[3] == native.ACT_GROUPED
        start = 0
        for g, (pname, kids) in enumerate(groups[L - 1]):
            assert tab[4 + 2 * M + g] == start and tab[4 + 3 * M + g] == len(kids)
            assert tab[4 + 4 * M + g] == levels[L - 1].index(pname)
            for k in range(start, start + len(kids)):
                assert tab[4 + k] == levels[L - 1].index(pname) and tab[4 + M + k] == g
                assert parent_of[levels[L][k]] == pname
            start += len(kids)


def test_product_never_imports_the_oracle():
    """The product path must not route through oracle/ (or the reference): scan every product module."""
    offenders = []
    for base, _, files in os.walk(PKG):
        for f in files:
            if not f.endswith(".py"):
                continue
            path = os.path.join(base, f)
            tree = ast.parse(open(path).read())
            for node in ast.walk(tree):
                names = []
                if isinstance(node, ast.Import):
                    names = [a.name for a in node.names]
                elif isinstance(node, ast.ImportFrom):
                    names = [node.module or ""]
                for n in names:
                    if n.split(".")[0] in ("oracle", "tests", "ref_shim") or "reference" in n:
                        offenders.append((path, n))
    assert not offenders, offenders
    for f in os.listdir(os.path.join(PKG, "csrc")):
        assert "oracle" not in open(os.path.join(PKG, "csrc", f)).read()


def test_dropin_module_surface():
    """Names / signatures train.py and predictEval.py rely on (SURVEY.md 8(b))."""
    import inspect
    from rhseg_b200.Metrics import losses, performance_metrics as pm
    from rhseg_b200.Models import models
    import rhseg_b200.tree_util as tu
    assert list(inspect.signature(models.UNet.__init__).parameters)[1:] == ["size", "n_channels", "hierarchy", "model_type"]
    assert list(inspect.signature(models.UNet.forward).parameters)[1:] == ["x", "type", "hierarchy", "threshold"]
    assert list(inspect.signature(models.HighResolutionNet.__init__).parameters)[1:4] == ["config", "hierarchy", "model_type"]
    for cls in (losses.CrossEntropyLoss, losses.SoftDiceLoss):
        assert list(inspect.signature(cls.forward).parameters)[1:] == ["outs", "targets", "logits_input", "class_weight"]
    assert list(inspect.signature(losses.hierarchical_consistency_loss).parameters) == ["probs_per_level", "levels", "parent_of", "reduction"]
    for cls in (pm.Accuracy, pm.Jaccardindex, pm.DiceScore, pm.Precision, pm.Recall):
        assert list(inspect.signature(cls.forward).parameters)[1:] == ["probs", "targets", "device", "num_classes", "child_classes"]
    for name in ("node", "create_tree_from_textfile", "add_channels", "add_levels", "find_depth", "getTreeList", "update_channels"):
        assert hasattr(tu, name)
    m = models.UNet(size=64, n_channels=3, hierarchy=EXT, model_type=1)
    keys = set(m.state_dict())
    assert {"heads.3.conv.weight", "films.2.mlp.1.bias", "inc0.conv.conv.0.weight", "up4.conv.conv.4.running_var",
            "down1.mpconv.1.conv.3.weight"} <= keys
    assert tuple(m.state_dict()["films.2.mlp.1.weight"].shape) == (128, 4)
    assert m.levels == O.hierarchy_tables(EXT)[0] and m.child_groups == O.hierarchy_tables(EXT)[3]
    flat = models.UNet(size=64, n_channels=1, hierarchy=EXT, model_type=0)
    assert flat.out_flat.conv.out_channels == 7
    with pytest.raises(Exception):
        m(torch.zeros(1, 3, 32, 32), type=1)  # CPU tensors: the head refuses loudly, no fallback


def test_text_tree_utilities(tmp_path):
    import rhseg_b200.tree_util as tu
    p = tmp_path / "tree.txt"
    p.write_text("background\nupper\ntooth\n\tpulp\n\tdentin\n\t\tinner\nlower\n")
    root = tu.create_tree_from_textfile(str(p))
    assert [c.name for c in root.children] == ["background", "upper", "tooth", "lower"]
    assert [c.name for c in root.children[2].children] == ["pulp", "dentin"]
    assert tu.find_depth(root) == 3
    assert tu.add_channels(root, 0) == 5
    tu.add_levels(root, tu.find_depth(root))
    # values verified against the reference's tree_util.py on the same file (build container)
    assert tu.getTreeList(root) == [[[0], [1], [2], [3], [4]], [[0], [1], [2], [3], [4]], [[0], [1], [2, 3], [4]]]
    assert [c.level for c in root.children] == [2, 2, 2, 2] and root.children[2].children[1].children[0].level == 0


def test_bench_byte_model_matches_survey():
    import bench
    wl = bench.WORKLOADS["unet_tl_620_b4"]
    alg = bench.algorithmic_bytes(wl, 4)
    assert abs(alg["step"] / 1e9 - 2.669) < 0.002 and abs(alg["metrics"] / 1e9 - 0.098) < 0.001
    wl = bench.WORKLOADS["hrnet_w48_tl_620_b4"]
    alg = bench.algorithmic_bytes(wl, 4)
    assert abs(alg["step"] / 1e9 - 1.968) < 0.002
    wl = bench.WORKLOADS["hrnet_w48_ext_620_b4"]
    alg = bench.algorithmic_bytes(wl, 4)
    assert abs(alg["step"] / 1e9 - 3.776) < 0.003
    assert bench.tree_shape(wl)[2:] == ([2, 2, 4, 3], [0, 1, 2, 1])
    alg = bench.algorithmic_bytes(bench.WORKLOADS["flat7_620_b4"], 4)   # SURVEY 8(d) row 4: 140 B/px + 56 B/px metrics
    assert abs(alg["step"] / 1e9 - 0.215) < 0.001 and abs(alg["metrics"] / 1e9 - 0.086) < 0.001
    alg = bench.algorithmic_bytes(bench.WORKLOADS["unet_tl_1024_b64"], 64)  # row 5: 116.5 GB in total
    assert abs(alg["step"] / 1e9 - 116.5) < 0.1


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _dist_worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from oracle import hier_oracle as Or
    from rhseg_b200 import dist as rdist
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    try:
        levels, parent_of, _, groups = Or.hierarchy_tables(TL)
        g = torch.Generator().manual_seed(0)
        B, H, W = 4, 12, 10
        logits = [torch.randn(B, 4, H, W, generator=g) for _ in range(2)]
        targets = Or.synth_targets(levels, groups, B, H, W, g)
        targets[1][1] = -1.0  # one sample without any valid child pixel: dice NaN there, CE -> 1.0
        weights = [[0.3, 1.5, 0.9, 0.2], [1.5, 0.3, 1.0, 3.9]]
        lo, hi = rdist.shard_batch(B, rank, world)

        def summary(zs, ts):
            onehots, evals = Or.predict_onehot_masked(zs, ts)
            n = len(zs)
            scal = torch.zeros(2 + 4 * n)
            scal[1] = Or.consistency_loss(onehots, levels, parent_of)
            conf = []
            for L in range(n):
                ce = Or.ce_loss(zs[L], ts[L], weights[L])
                per = [Or.dice_loss(zs[L][i:i + 1], ts[L][i:i + 1], weights[L]) for i in range(zs[L].shape[0])]
                valid = [d for d in per if d is not None]
                scal[2 + 4 * L] = ce
                scal[3 + 4 * L] = torch.stack(valid).mean() if valid else 0.0
                scal[4 + 4 * L] = len(valid)
                scal[5 + 4 * L] = zs[L].shape[0]
                conf.append(Or.level_confusion(onehots[L], evals[L], 4, L != 0))
            scal[0] = scal[1] + sum(scal[2 + 4 * L] + scal[3 + 4 * L] for L in range(n))
            return scal, conf

        scal, conf = summary([z[lo:hi] for z in logits], [t[lo:hi] for t in targets])
        got = rdist.all_reduce_step_summary(scal, hi - lo, conf)
        ref_scal, ref_conf = summary(logits, targets)
        ok = abs(float(got["total"]) - float(ref_scal[0])) < 1e-5
        ok &= all(torch.equal(a, b) for a, b in zip(got["confusion"], ref_conf))
        ok &= abs(float(got["dice"][1]) - float(ref_scal[3 + 4])) < 1e-6 and float(got["n_dice"][1]) == 3.0
        scale = rdist.dice_grad_scale(scal[4 + 4].double(), got["n_dice"][1], world)
        # exchange-buffer form ([summary | parameter gradients], one all-reduce): host logic on CPU tensors
        summ = rdist.pack_step_summary(scal, hi - lo, conf)
        grads = [torch.full((3, 2), float(rank + 1)), torch.arange(5, dtype=torch.float32) * (rank + 1)]
        buf = rdist.pack_exchange(summ, grads)
        ok &= buf.dtype == torch.float64 and buf.numel() == summ.numel() + 11
        dist.all_reduce(buf)
        back = [torch.zeros(3, 2), torch.zeros(5)]
        rdist.unpack_exchange(buf, summ.numel(), back, scale=1.0 / world)
        ok &= bool(torch.equal(back[0], torch.full((3, 2), 1.5))) and bool(torch.equal(back[1], torch.arange(5, dtype=torch.float32) * 1.5))
        glob = rdist.unpack_global(buf, len(logits), [tuple(c.shape) for c in conf])
        ok &= abs(float(glob["total"]) - float(ref_scal[0])) < 1e-5
        try:  # the peer-memory exchange is CUDA-only and says so
            rdist.PeerExchange(16)
            ok = False
        except Exception as e:
            ok &= "NativeError" in type(e).__name__ or "CUDA" in str(e) or "cuda" in str(e)
        q.put((rank, bool(ok), float(scale)))
    finally:
        dist.destroy_process_group()


def test_batch_sharded_summary_exchange_gloo_world2(monkeypatch):
    import torch.multiprocessing as mp
    # host logic: the workers see no GPU, also on a machine that has one (they check that PeerExchange refuses to run)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dist_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=180) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert [r[1] for r in res] == [True, True], res
    # rank 0 holds samples 0-1 (sample 1 has no valid dice) -> 1 of 3 valid; rank 1 holds 2 of 3
    assert abs(res[0][2] - 2 * 1 / 3) < 1e-9 and abs(res[1][2] - 2 * 2 / 3) < 1e-9


def test_reference_arm_prints_the_contract_line():
    """bench.py --impl reference (CPU only): one JSON line, the same `config` object as our arm would print for the same
    command line, the reference's own modules when they are staged (kind "reference"), the oracle port otherwise."""
    import json
    import subprocess
    import bench
    from oracle import ref_loader
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "flat7_620_b4",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "Mpixel/s" and line["higher_is_better"] is True
    assert line["config"] == bench.config_of("flat7_620_b4", bench.WORKLOADS["flat7_620_b4"], 1)
    assert line["cpu_baseline"]["kind"] == ("reference" if ref_loader.available() else "port")
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["value"] > 0
