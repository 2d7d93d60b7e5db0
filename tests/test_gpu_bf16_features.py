"""bf16 donor features (backbones trained under torch.autocast) through the hierarchical head and the fused step.

Contract (DESIGN.md 3.7): with bf16 features the kernels compute what the fp32 path computes on feats.float() -- each
value is converted to fp32 exactly, every sum, activation, loss, metric and parameter gradient stays fp32 / fp64 -- and
dfeats is formed in fp32 and rounded to bf16 once, when stored.  So the reference of every check here is the fp32 path
on the upcast features.  The dtype checks at the bottom run without a GPU."""
import pytest
import torch

from helpers import HIER_CASES, Fixture, close
from oracle import hier_oracle as O
from test_gpu_shapes import CASES as SHAPE_CASES
from test_gpu_shapes import _inputs as shape_inputs

DEV = "cuda"
BF = torch.bfloat16
gpu = pytest.mark.gpu


def close_dfeats(got, ref, what="", roundings=1):
    """bf16 dfeats against the fp32 path's dfeats: one bf16 rounding (2^-8 relative) plus fp32 reordering.
    roundings=2: against another bf16 result (each side rounded once)."""
    assert got.dtype == BF, (what, got.dtype)
    a, r = got.detach().double().cpu(), ref.detach().double().cpu()
    bound = roundings * 2.0 ** -8 * r.abs() + 1e-5 * r.abs().max() + 1e-12
    bad = (a - r).abs() > bound
    assert not bad.any(), "%s: %d/%d out of tolerance, max err %.3e" % (what, int(bad.sum()), r.numel(), (a - r).abs().max())


def min_top2_margin(z):
    if z.shape[1] < 2:
        return float("inf")
    top = z.detach().float().topk(2, dim=1).values
    return (top[:, 0] - top[:, 1]).min().item()


def _fx_leaves(fx, dtype):
    mk = lambda ts: [t.to(DEV).requires_grad_(True) for t in ts]
    feats = [t.to(BF).to(dtype).to(DEV).requires_grad_(True) for t in fx.per_level("feats")]
    hw, hb = mk(fx.per_level("head_w")), mk(fx.per_level("head_b"))
    fw, fb = mk(fx.per_level("film_w", n=fx.nL - 1)), mk(fx.per_level("film_b", n=fx.nL - 1))
    target = torch.cat(fx.per_level("target"), dim=1).to(DEV)
    return feats, hw, hb, fw, fb, target


def _compare_steps(name, out, ref, leaves, ref_leaves, targets, nL, rtol_z=1e-5):
    from rhseg_b200 import metric_ops
    assert out.loss.dtype == torch.float32 and out.scalars.dtype == torch.float32
    close(out.scalars, ref.scalars, what=f"{name} loss / consistency / per-level CE, Dice")
    for L in range(nL):
        assert out.logits[L].dtype == torch.float32 and out.probs[L].dtype == torch.float32
        close(out.logits[L], ref.logits[L], rtol=rtol_z, what=f"{name} logits{L}")
        close(out.probs[L], ref.probs[L], rtol=rtol_z, what=f"{name} probs{L}")
        assert out.confusion[L].dtype == torch.int64
        own = metric_ops.confusion_from_logits(out.logits[L].detach(), targets[L], L != 0)
        assert torch.equal(out.confusion[L], own), f"{name} confusion{L} vs its own logits"
        if min_top2_margin(ref.logits[L]) >= 1e-5:
            assert torch.equal(out.confusion[L], ref.confusion[L]), f"{name} confusion{L} vs the fp32 path"
    feats, ref_feats = leaves[0], ref_leaves[0]
    for L in range(nL):
        close_dfeats(feats[L].grad, ref_feats[L].grad, what=f"{name} dfeats{L}")
    for grp, rgrp, nm in zip(leaves[1:], ref_leaves[1:], ("dhead_w", "dhead_b", "dfilm_w", "dfilm_b")):
        for i, (a, b) in enumerate(zip(grp, rgrp)):
            assert a.grad.dtype == torch.float32
            close(a.grad, b.grad, what=f"{name} {nm}{i}")


# ------------------------------------------------------------------------------------------------------------------
# fused step on every head fixture
# ------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", HIER_CASES)
def test_fused_step_bf16_equals_fp32_on_upcast_features(name):
    import rhseg_b200
    fx = Fixture(name)
    step = rhseg_b200.FusedHierStep(fx.tree, fx.level_weights)
    *leaves, target = _fx_leaves(fx, BF)
    *ref_leaves, _ = _fx_leaves(fx, torch.float32)
    out = step(*leaves, target, fx.out_size)
    out.loss.backward()
    ref = step(*ref_leaves, target, fx.out_size)
    ref.loss.backward()
    targets = [t.to(DEV) for t in fx.per_level("target")]
    # 720-channel donors: the bf16 forward splits pixel tiles differently (2e-5, as tests/test_gpu_fullsize.py documents)
    _compare_steps(name, out, ref, leaves, ref_leaves, targets, fx.nL, rtol_z=2e-5 if fx.kind == "hrnet" else 1e-5)


# ------------------------------------------------------------------------------------------------------------------
# ragged shapes (tests/test_gpu_shapes.py): odd planes, C not a multiple of the stage, K = 8, non-integer upsampling
# ------------------------------------------------------------------------------------------------------------------
def _shape_leaves(tensors, dtype, offset=0):
    feats = []
    for f in tensors[0]:
        fb = f.to(BF).to(dtype)
        if offset:  # a slice of a larger buffer: the base pointer sits `offset` elements past a 16-byte boundary
            buf = torch.zeros(fb.numel() + 16, dtype=dtype, device=DEV)
            assert buf.data_ptr() % 16 == 0
            v = buf[offset:offset + fb.numel()].view(fb.shape)
            v.copy_(fb)
            feats.append(v.requires_grad_(True))
        else:
            feats.append(fb.to(DEV).requires_grad_(True))
    rest = [[t.clone().to(DEV).requires_grad_(True) for t in grp] for grp in tensors[1:]]
    return [feats] + rest


def _run_shape_case(case, offset=0):
    import rhseg_b200
    name, tree_dict, B, C, h, w, out_size = case
    levels, parent_of, groups, chans, tensors, targets, weights = shape_inputs(tree_dict, B, C, h, w, out_size, seed=len(name))
    n = len(chans)
    step = rhseg_b200.FusedHierStep(tree_dict, weights)
    target = torch.cat(targets, dim=1).to(DEV)
    tg = [t.to(DEV) for t in targets]
    leaves = _shape_leaves(tensors, BF, offset)
    if offset:
        assert leaves[0][0].data_ptr() % 16 == 2 * offset
    ref_leaves = _shape_leaves(tensors, torch.float32)
    out = step(*leaves, target, out_size)
    out.loss.backward()
    ref = step(*ref_leaves, target, out_size)
    ref.loss.backward()
    _compare_steps(f"{name}@{offset}", out, ref, leaves, ref_leaves, tg, n)
    # the drop-in head on the same inputs
    tree = rhseg_b200.ClassTree(tree_dict)
    leaves = _shape_leaves(tensors, BF, offset)
    ref_leaves = _shape_leaves(tensors, torch.float32)
    gen = torch.Generator().manual_seed(3)
    probs, logits = rhseg_b200.hier_head_forward(tree, *leaves, out_size)
    probs_r, logits_r = rhseg_b200.hier_head_forward(tree, *ref_leaves, out_size)
    wz = [torch.randn(z.shape, generator=gen).to(DEV) for z in logits]
    wp = [torch.randn(p.shape, generator=gen).to(DEV) for p in probs]
    sum(((z * a).sum() + (p * b).sum()) for z, p, a, b in zip(logits, probs, wz, wp)).backward()
    sum(((z * a).sum() + (p * b).sum()) for z, p, a, b in zip(logits_r, probs_r, wz, wp)).backward()
    for L in range(n):
        close(logits[L], logits_r[L], what=f"{name}@{offset} head logits{L}")
        close(probs[L], probs_r[L], what=f"{name}@{offset} head probs{L}")
        close_dfeats(leaves[0][L].grad, ref_leaves[0][L].grad, what=f"{name}@{offset} head dfeats{L}")
    for grp, rgrp in zip(leaves[1:], ref_leaves[1:]):
        for a, b in zip(grp, rgrp):
            close(a.grad, b.grad, what=f"{name}@{offset} head parameter gradient")


@gpu
@pytest.mark.parametrize("case", SHAPE_CASES, ids=[c[0] for c in SHAPE_CASES])
def test_ragged_shapes_bf16_equal_fp32_on_upcast_features(case):
    _run_shape_case(case)


@gpu
@pytest.mark.parametrize("offset", range(1, 8))
@pytest.mark.parametrize("case", [SHAPE_CASES[0], SHAPE_CASES[2], SHAPE_CASES[3]], ids=lambda c: c[0])
def test_feature_base_at_every_2_byte_offset(case, offset):
    """bf16 rows start anywhere inside a 16-byte granule: producer shifts 0..7, with even (vector rows) and odd planes."""
    _run_shape_case(case, offset)


# ------------------------------------------------------------------------------------------------------------------
# drop-in models under autocast
# ------------------------------------------------------------------------------------------------------------------
TL = {"background": {}, "upper": {}, "lower": {}, "tooth": {"pulp": {}, "dentin": {}, "enamel": {}, "composite": {}}}


def _small_hrnet_config():
    from oracle import ref_loader
    st = lambda blocks, ch, block="BASIC": {"NUM_MODULES": 1, "NUM_BRANCHES": len(ch), "BLOCK": block, "NUM_BLOCKS": blocks,
                                            "NUM_CHANNELS": ch, "FUSE_METHOD": "SUM"}
    return ref_loader.CfgNode({"MODEL": {"ALIGN_CORNERS": True, "EXTRA": {
        "FINAL_CONV_KERNEL": 1, "STAGE1": st([1], [16], "BOTTLENECK"), "STAGE2": st([1, 1], [8, 16]),
        "STAGE3": st([1, 1, 1], [8, 16, 32]), "STAGE4": st([1, 1, 1, 1], [8, 16, 32, 64])}}})


@gpu
@pytest.mark.parametrize("donor", ["unet", "hrnet"])
def test_dropin_models_train_under_autocast(donor):
    import rhseg_b200
    from rhseg_b200.Models import models
    torch.manual_seed(7)
    if donor == "unet":
        m = models.UNet(size=32, n_channels=3, hierarchy=TL, model_type=1).to(DEV)
        x = torch.randn(2, 3, 32, 40, device=DEV)
        run = lambda: m(x, type=1, hierarchy=TL)
    else:
        m = models.HighResolutionNet(_small_hrnet_config(), hierarchy=TL, model_type=1).to(DEV)
        x = torch.randn(2, 3, 36, 44, device=DEV)  # feature plane 9 x 11: odd
        run = lambda: m(x)
    m.train()
    seen = {}
    inner = m._head_forward

    def spy(feats, head_convs, out_size=None):
        seen["feats"] = [f.detach().clone() for f in feats]
        return inner(feats, head_convs, out_size)

    m._head_forward = spy
    with torch.autocast("cuda", dtype=torch.bfloat16):
        probs, logits = run()
    assert all(f.dtype == BF for f in seen["feats"]), [f.dtype for f in seen["feats"]]
    assert all(z.dtype == torch.float32 for z in logits) and all(p.dtype == torch.float32 for p in probs)
    # outputs = the head on the upcast features with the model's own parameters
    n = len(logits)
    heads = [h.conv for h in m.heads] if donor == "unet" else list(m.classifiers)
    lin = [f.mlp[1] for f in m.films]
    with torch.no_grad():
        p_ref, z_ref = rhseg_b200.hier_head_forward(m._tree, [f.float() for f in seen["feats"]], [c.weight for c in heads],
                                                    [c.bias for c in heads], [l.weight for l in lin], [l.bias for l in lin],
                                                    None if donor == "unet" else tuple(x.shape[-2:]))
    for L in range(n):
        close(logits[L], z_ref[L], what=f"{donor} logits{L}")
        close(probs[L], p_ref[L], what=f"{donor} probs{L}")
    loss = sum(z.square().mean() + p.mean() for z, p in zip(logits, probs))
    loss.backward()
    for nm, p in m.named_parameters():
        assert p.grad is not None, nm
        assert torch.isfinite(p.grad).all(), nm


# ------------------------------------------------------------------------------------------------------------------
# CUDA graph, data parallel, launch count
# ------------------------------------------------------------------------------------------------------------------
@gpu
def test_bf16_step_replays_from_a_cuda_graph():
    import rhseg_b200
    fx = Fixture("hrnet_tl")
    step = rhseg_b200.FusedHierStep(fx.tree, fx.level_weights)
    feats, hw, hb, fw, fb, target = _fx_leaves(fx, BF)
    params = [hw, hb, fw, fb]
    leaves = feats + [p for grp in params for p in grp]
    one = torch.ones((), device=DEV)

    def run():
        out = step(feats, *params, target, fx.out_size)
        return out, torch.autograd.grad(out.loss, leaves, grad_outputs=one)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            run()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_out, g_grads = run()
    gen = torch.Generator().manual_seed(5)
    for it in range(2):
        with torch.no_grad():
            for f in feats:
                f.copy_(torch.randn(f.shape, generator=gen).to(BF))
            params[0][0].mul_(0.9)
        graph.replay()
        torch.cuda.synchronize()
        got = (g_out.loss.clone(), [c.clone() for c in g_out.confusion], [g.clone() for g in g_grads])
        e_out, e_grads = run()
        torch.cuda.synchronize()
        close(got[0], e_out.loss, what="graph loss %d" % it)
        for a, b in zip(got[1], e_out.confusion):
            assert torch.equal(a, b)
        for i, (a, b) in enumerate(zip(got[2], e_grads)):
            assert a.dtype == b.dtype
            if a.dtype == BF:  # the order of fp64 atomics may move an fp32 value across a bf16 rounding boundary
                close_dfeats(a, b.float(), what="graph dfeats %d/%d" % (it, i), roundings=2)
            else:
                close(a, b, rtol=1e-6, what="graph grad %d/%d" % (it, i))


@gpu
@pytest.mark.parametrize("name,shards", [("unet_tl_odd_notooth", [slice(0, 1), slice(1, 3)]),
                                         ("hrnet_ext", [slice(0, 1), slice(1, 2)])])
def test_sharded_bf16_step_equals_the_whole_batch(name, shards):
    import rhseg_b200
    fx = Fixture(name)
    world = len(shards)
    step = rhseg_b200.FusedHierStep(fx.tree, fx.level_weights)

    def leaves(sl=slice(None)):
        feats, hw, hb, fw, fb, target = _fx_leaves(fx, BF)
        feats = [f.detach()[sl].contiguous().requires_grad_(True) for f in feats]
        return feats, hw, hb, fw, fb, target[sl].contiguous()

    feats, hw, hb, fw, fb, target = leaves()
    whole = step(feats, hw, hb, fw, fb, target, fx.out_size)
    whole.loss.backward()
    want_params = [p.grad.clone() for grp in (hw, hb, fw, fb) for p in grp]
    want_dfeats = [f.grad.float() for f in feats]
    gsum = torch.stack([step(*leaves(sl), fx.out_size).summary.clone() for sl in shards]).sum(0)
    step.data_parallel(lambda s: gsum.clone(), world)
    acc = [torch.zeros_like(g) for g in want_params]
    try:
        for sl in shards:
            f, a, b, c, d, t = leaves(sl)
            out = step(f, a, b, c, d, t, fx.out_size)
            out.loss.backward()
            for dst, p in zip(acc, [p for grp in (a, b, c, d) for p in grp]):
                dst += p.grad / world
            for L in range(fx.nL):
                close_dfeats(f[L].grad / world, want_dfeats[L][sl], what=f"{name} dfeats{L} shard {sl}", roundings=2)
    finally:
        step.data_parallel(None, 1)
    for got, want in zip(acc, want_params):
        close(got, want, what=f"{name} parameter gradient")


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return sorted(n.split("<")[0] for n in names)  # template arguments (the feature type) aside


@gpu
@pytest.mark.parametrize("name", ["unet_tl", "hrnet_tl"])
def test_bf16_step_launches_what_the_fp32_step_launches(name):
    """No hidden cast: the bf16 step (forward + backward) runs the same kernels as the fp32 step, no copy or conversion."""
    import rhseg_b200
    fx = Fixture(name)
    step = rhseg_b200.FusedHierStep(fx.tree, fx.level_weights)
    runs = {}
    for dt in (torch.float32, BF):
        feats, hw, hb, fw, fb, target = _fx_leaves(fx, dt)
        leaves = feats + hw + hb + fw + fb

        def one_step():
            out = step(feats, hw, hb, fw, fb, target, fx.out_size)
            torch.autograd.grad(out.loss, leaves)

        one_step()  # warm: tables, workspaces
        runs[dt] = _kernel_names(one_step)
    assert runs[BF] == runs[torch.float32], (runs[BF], runs[torch.float32])
    assert not any("copy" in n.lower() or "convert" in n.lower() for n in runs[BF]), runs[BF]


# ------------------------------------------------------------------------------------------------------------------
# dtype validation (no GPU needed: raised before the device check)
# ------------------------------------------------------------------------------------------------------------------
def _cpu_head_inputs(feat_dtypes, param_dtype=torch.float32):
    import rhseg_b200
    tree = rhseg_b200.ClassTree(TL)
    C = 8
    feats = [torch.zeros(1, C, 4, 4, dtype=dt) for dt in feat_dtypes]
    hw = [torch.zeros(k, C, 1, 1, dtype=param_dtype) for k in tree.head_channels]
    hb = [torch.zeros(k, dtype=param_dtype) for k in tree.head_channels]
    fw = [torch.zeros(2 * C, tree.head_channels[0], dtype=param_dtype)]
    fb = [torch.zeros(2 * C, dtype=param_dtype)]
    return tree, feats, hw, hb, fw, fb


@pytest.mark.parametrize("feat_dtypes,param_dtype,needle", [
    ((torch.float16, torch.float16), torch.float32, "bfloat16"),        # fp16 features: loss scaling is a separate matter
    ((torch.float32, torch.bfloat16), torch.float32, "one dtype"),      # mixed levels
    ((torch.bfloat16, torch.bfloat16), torch.bfloat16, "float32"),      # parameters stay fp32
    ((torch.float64, torch.float64), torch.float32, "bfloat16"),
])
def test_feature_and_parameter_dtypes_are_validated(feat_dtypes, param_dtype, needle):
    import rhseg_b200
    from rhseg_b200 import native
    tree, feats, hw, hb, fw, fb = _cpu_head_inputs(feat_dtypes, param_dtype)
    with pytest.raises(native.NativeError, match=needle):
        rhseg_b200.hier_head_forward(tree, feats, hw, hb, fw, fb)


def test_bf16_cpu_features_reach_the_device_check():
    """Accepted dtypes pass validation and fail only because there is no CPU path."""
    import rhseg_b200
    from rhseg_b200 import native
    tree, feats, hw, hb, fw, fb = _cpu_head_inputs((torch.bfloat16, torch.bfloat16))
    with pytest.raises(native.NativeError, match="CUDA"):
        rhseg_b200.hier_head_forward(tree, feats, hw, hb, fw, fb)
