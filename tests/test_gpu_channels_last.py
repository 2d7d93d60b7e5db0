"""Channels-last donor features (models converted with torch.channels_last) through the hierarchical head and the fused
step, read in place by the NHWC kernels (RHSEG_FEATS_NHWC).

Contract (DESIGN.md 3.8): the reference of every check is the same step on the same values in contiguous (NCHW) form.
At feature resolution (UNet) logits, probabilities and confusion matrices are bit-identical; dfeats is bit-identical for
the same dz (the conv backward forms every element in the NCHW kernel's order), and in the full step it agrees to the
1e-5 tolerance where dz carries the FiLM pool gradient of the next level (formed from the fp64 sums S / s, which both
paths add in different orders).  Upsampled heads (HRNet): logits within 1e-5.  dfeats comes back channels-last.  The
checks at the bottom run without a GPU."""
import os
import re

import pytest
import torch

from helpers import HIER_CASES, Fixture, close
from test_gpu_shapes import CASES as SHAPE_CASES
from test_gpu_shapes import _inputs as shape_inputs

DEV = "cuda"
BF = torch.bfloat16
CL = torch.channels_last
gpu = pytest.mark.gpu
DTYPES = [torch.float32, BF]
DT_IDS = ["fp32", "bf16"]


def is_cl(t):
    return t.is_contiguous(memory_format=CL) and not t.is_contiguous()


def _cl_leaf(t, dtype):
    return t.to(dtype).to(DEV).contiguous(memory_format=CL).requires_grad_(True)


def _nchw_leaf(t, dtype):
    return t.to(dtype).to(DEV).contiguous().requires_grad_(True)


def _fx_leaves(fx, dtype, layout):
    mk = lambda ts: [t.to(DEV).requires_grad_(True) for t in ts]
    conv = _cl_leaf if layout == "cl" else _nchw_leaf
    feats = [conv(t.to(BF) if dtype == BF else t, dtype) for t in fx.per_level("feats")]
    hw, hb = mk(fx.per_level("head_w")), mk(fx.per_level("head_b"))
    fw, fb = mk(fx.per_level("film_w", n=fx.nL - 1)), mk(fx.per_level("film_b", n=fx.nL - 1))
    target = torch.cat(fx.per_level("target"), dim=1).to(DEV)
    return feats, hw, hb, fw, fb, target


def _compare(name, out, ref, leaves, ref_leaves, nL, fullres, native_cl):
    """fused-step outputs and gradients of the channels-last run (out, leaves) against the contiguous run"""
    close(out.scalars, ref.scalars, what=f"{name} loss / consistency / per-level CE, Dice")
    for L in range(nL):
        if fullres:
            assert torch.equal(out.logits[L], ref.logits[L]), f"{name} logits{L}"
            assert torch.equal(out.probs[L], ref.probs[L]), f"{name} probs{L}"
            assert torch.equal(out.confusion[L], ref.confusion[L]), f"{name} confusion{L}"
        else:
            close(out.logits[L], ref.logits[L], what=f"{name} logits{L}")
            close(out.probs[L], ref.probs[L], what=f"{name} probs{L}")
    _compare_grads(name, leaves, ref_leaves, nL, fullres, native_cl)


def _compare_grads(name, leaves, ref_leaves, nL, fullres, native_cl):
    feats, ref_feats = leaves[0], ref_leaves[0]
    for L in range(nL):
        g, r = feats[L].grad, ref_feats[L].grad
        assert g.dtype == r.dtype
        if native_cl:
            assert is_cl(g), f"{name} dfeats{L} is not channels-last: strides {g.stride()}"
        # the last level's dz has no FiLM successor: the same inputs in both runs
        if fullres and L == nL - 1:
            assert torch.equal(g, r), f"{name} dfeats{L}"
        elif g.dtype == BF:  # an fp32 value a few ulp apart may round to the neighbouring bf16
            a, b = g.double().cpu(), r.double().cpu()
            bad = (a - b).abs() > 2.0 ** -7 * b.abs() + 1e-5 * b.abs().max() + 1e-12
            assert not bad.any(), f"{name} dfeats{L}: {int(bad.sum())} out of tolerance"
        else:
            close(g, r, what=f"{name} dfeats{L}")
    for grp, rgrp, nm in zip(leaves[1:], ref_leaves[1:], ("dhead_w", "dhead_b", "dfilm_w", "dfilm_b")):
        for i, (a, b) in enumerate(zip(grp, rgrp)):
            close(a.grad, b.grad, what=f"{name} {nm}{i}")


def _native(feats):
    from rhseg_b200 import head
    return all(head._nhwc_native(f) for f in feats)


# ------------------------------------------------------------------------------------------------------------------
# every head fixture, fused step and drop-in head
# ------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("name", HIER_CASES)
def test_fused_step_channels_last_equals_contiguous(name, dtype):
    import rhseg_b200
    fx = Fixture(name)
    step = rhseg_b200.FusedHierStep(fx.tree, fx.level_weights)
    *leaves, target = _fx_leaves(fx, dtype, "cl")
    *ref_leaves, _ = _fx_leaves(fx, dtype, "nchw")
    assert all(is_cl(f) for f in leaves[0]) and _native(leaves[0])
    out = step(*leaves, target, fx.out_size)
    out.loss.backward()
    ref = step(*ref_leaves, target, fx.out_size)
    ref.loss.backward()
    _compare(f"{name}/{dtype}", out, ref, leaves, ref_leaves, fx.nL, fx.kind == "unet", True)


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("name", HIER_CASES)
def test_dropin_head_channels_last_equals_contiguous(name, dtype):
    import rhseg_b200
    fx = Fixture(name)
    tree = rhseg_b200.ClassTree(fx.tree)
    *leaves, _ = _fx_leaves(fx, dtype, "cl")
    *ref_leaves, _ = _fx_leaves(fx, dtype, "nchw")
    probs, logits = rhseg_b200.hier_head_forward(tree, *leaves, fx.out_size)
    probs_r, logits_r = rhseg_b200.hier_head_forward(tree, *ref_leaves, fx.out_size)
    fullres = fx.kind == "unet"
    for L in range(fx.nL):
        if fullres:
            assert torch.equal(logits[L], logits_r[L]) and torch.equal(probs[L], probs_r[L]), f"{name} level {L}"
        else:
            close(logits[L], logits_r[L], what=f"{name} logits{L}")
            close(probs[L], probs_r[L], what=f"{name} probs{L}")
    gen = torch.Generator().manual_seed(3)
    wz = [torch.randn(z.shape, generator=gen).to(DEV) for z in logits]
    wp = [torch.randn(p.shape, generator=gen).to(DEV) for p in probs]
    sum(((z * a).sum() + (p * b).sum()) for z, p, a, b in zip(logits, probs, wz, wp)).backward()
    sum(((z * a).sum() + (p * b).sum()) for z, p, a, b in zip(logits_r, probs_r, wz, wp)).backward()
    _compare_grads(name, leaves, ref_leaves, fx.nL, fullres, True)


# ------------------------------------------------------------------------------------------------------------------
# the conv backward alone: dfeats bit-identical for the same dz
# ------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("B,C,h,w,K", [(3, 64, 16, 20, 4), (2, 720, 13, 11, 4), (1, 64, 7, 9, 3), (2, 16, 5, 7, 8),
                                       (2, 720, 31, 31, 1), (1, 40, 33, 3, 5)])
def test_conv_backward_dfeats_bit_identical(B, C, h, w, K, dtype):
    from rhseg_b200 import native
    from rhseg_b200.native import call, ptr, stream_of
    g = torch.Generator().manual_seed(B * 1000 + C + K)
    x = torch.randn(B, C, h, w, generator=g).to(dtype).to(DEV)
    dz = torch.randn(B, K, h, w, generator=g).to(DEV)
    ew = (torch.randn(B, K, C, generator=g) * 0.3).to(DEV)
    bf = native.FEATS_BF16 if dtype == BF else 0
    res = {}
    for layout, f in (("nchw", x.contiguous()), ("cl", x.contiguous(memory_format=CL))):
        df = torch.empty_like(f)
        S = torch.zeros(B, K, C, dtype=torch.float64, device=DEV)
        s = torch.zeros(B, K, dtype=torch.float64, device=DEV)
        call("rhseg_head_conv_bwd", ptr(f), ptr(dz), ptr(ew), B, C, K, h * w, ptr(df), ptr(S), ptr(s),
             bf | (native.FEATS_NHWC if layout == "cl" else 0), stream_of(f))
        res[layout] = (df, S, s)
    torch.cuda.synchronize()
    assert is_cl(res["cl"][0]) or C == 1
    assert torch.equal(res["cl"][0], res["nchw"][0])
    ref = torch.einsum("bkn,bcn->bkc", dz.double().view(B, K, -1), x.double().view(B, C, -1))
    close(res["cl"][1], ref, what="S")
    close(res["cl"][1], res["nchw"][1], what="S against NCHW")
    close(res["cl"][2], res["nchw"][2], what="s")


# ------------------------------------------------------------------------------------------------------------------
# ragged shapes and the fallback cases (tests/test_gpu_shapes.py): odd planes, B = 9, partial tiles, C not a multiple
# of 16 bytes (C = 33, C = 18, bf16 C = 20: the contiguous copy of today), non-integer upsampling
# ------------------------------------------------------------------------------------------------------------------
def _shape_run(case, dtype, make_feats):
    import rhseg_b200
    name, tree_dict, B, C, h, w, out_size = case
    levels, parent_of, groups, chans, tensors, targets, weights = shape_inputs(tree_dict, B, C, h, w, out_size, seed=len(name))
    step = rhseg_b200.FusedHierStep(tree_dict, weights)
    target = torch.cat(targets, dim=1).to(DEV)
    rest = lambda: [[t.clone().to(DEV).requires_grad_(True) for t in grp] for grp in tensors[1:]]
    src = [t.to(BF) if dtype == BF else t for t in tensors[0]]
    leaves = [make_feats(src, dtype)] + rest()
    ref_leaves = [[_nchw_leaf(t, dtype) for t in src]] + rest()
    out = step(*leaves, target, out_size)
    out.loss.backward()
    ref = step(*ref_leaves, target, out_size)
    ref.loss.backward()
    return name, out, ref, leaves, ref_leaves, len(chans), out_size is None


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("case", SHAPE_CASES, ids=[c[0] for c in SHAPE_CASES])
def test_ragged_shapes_channels_last(case, dtype):
    C = case[3]
    native_cl = (C * (2 if dtype == BF else 4)) % 16 == 0
    name, out, ref, leaves, ref_leaves, n, fullres = _shape_run(case, dtype, lambda src, dt: [_cl_leaf(t, dt) for t in src])
    assert _native(leaves[0]) == native_cl
    _compare(f"{name}/{dtype}", out, ref, leaves, ref_leaves, n, fullres, native_cl)


def _misaligned_cl(t, dtype):
    """a channels-last view whose base sits one element past a 16-byte boundary"""
    B, C, h, w = t.shape
    buf = torch.zeros(t.numel() + 16, dtype=dtype, device=DEV)
    v = buf[1:1 + t.numel()].view(B, h, w, C).permute(0, 3, 1, 2)
    with torch.no_grad():
        v.copy_(t.to(dtype))
    assert is_cl(v) and v.data_ptr() % 16 != 0
    return v.requires_grad_(True)


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("case", [SHAPE_CASES[0], SHAPE_CASES[2]], ids=lambda c: c[0])
def test_misaligned_channels_last_base_takes_the_copy(case, dtype):
    name, out, ref, leaves, ref_leaves, n, fullres = _shape_run(case, dtype, lambda src, dt: [_misaligned_cl(t, dt) for t in src])
    assert not _native(leaves[0])
    _compare(f"{name}/{dtype}", out, ref, leaves, ref_leaves, n, fullres, False)


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("case", [SHAPE_CASES[2], SHAPE_CASES[4]], ids=lambda c: c[0])
def test_mixed_layouts_across_levels(case, dtype):
    mk = lambda src, dt: [(_cl_leaf if L % 2 == 0 else _nchw_leaf)(t, dt) for L, t in enumerate(src)]
    name, out, ref, leaves, ref_leaves, n, fullres = _shape_run(case, dtype, mk)
    assert [is_cl(f) for f in leaves[0]] == [L % 2 == 0 for L in range(n)]
    _compare(f"{name}/{dtype}", out, ref, leaves, ref_leaves, n, fullres, False)
    for L in range(n):
        assert is_cl(leaves[0][L].grad) == (L % 2 == 0), f"dfeats{L} layout"


# ------------------------------------------------------------------------------------------------------------------
# drop-in models converted to channels_last, with and without bf16 autocast
# ------------------------------------------------------------------------------------------------------------------
TL = {"background": {}, "upper": {}, "lower": {}, "tooth": {"pulp": {}, "dentin": {}, "enamel": {}, "composite": {}}}


@gpu
@pytest.mark.parametrize("autocast", [False, True], ids=["fp32", "autocast_bf16"])
@pytest.mark.parametrize("donor", ["unet", "hrnet"])
def test_dropin_models_in_channels_last(donor, autocast):
    import rhseg_b200
    from rhseg_b200.Models import models
    from test_gpu_bf16_features import _small_hrnet_config
    torch.manual_seed(7)
    if donor == "unet":
        m = models.UNet(size=32, n_channels=3, hierarchy=TL, model_type=1).to(DEV)
        x = torch.randn(2, 3, 32, 40, device=DEV)
        run = lambda: m(x, type=1, hierarchy=TL)
    else:
        m = models.HighResolutionNet(_small_hrnet_config(), hierarchy=TL, model_type=1).to(DEV)
        x = torch.randn(2, 3, 36, 44, device=DEV)
        run = lambda: m(x)
    m = m.to(memory_format=CL)
    x = x.contiguous(memory_format=CL)
    m.train()
    seen = {}
    inner = m._head_forward

    def spy(feats, head_convs, out_size=None):
        seen["feats"] = list(feats)
        seen["copy"] = [f.detach().clone(memory_format=torch.preserve_format) for f in feats]
        return inner(feats, head_convs, out_size)

    m._head_forward = spy
    with torch.autocast("cuda", dtype=BF, enabled=autocast):
        probs, logits = run()
    feats = seen["feats"]
    assert all(is_cl(f) for f in feats), [f.stride() for f in feats]  # the donor hands over channels-last features
    assert all(f.dtype == (BF if autocast else torch.float32) for f in feats)
    assert _native(feats)
    n = len(logits)
    heads = [h.conv for h in m.heads] if donor == "unet" else list(m.classifiers)
    lin = [f.mlp[1] for f in m.films]
    with torch.no_grad():
        p_ref, z_ref = rhseg_b200.hier_head_forward(m._tree, [f.contiguous() for f in seen["copy"]], [c.weight for c in heads],
                                                    [c.bias for c in heads], [l.weight for l in lin], [l.bias for l in lin],
                                                    None if donor == "unet" else tuple(x.shape[-2:]))
    for L in range(n):
        if donor == "unet":
            assert torch.equal(logits[L], z_ref[L]) and torch.equal(probs[L], p_ref[L]), f"unet level {L}"
        else:
            close(logits[L], z_ref[L], what=f"{donor} logits{L}")
            close(probs[L], p_ref[L], what=f"{donor} probs{L}")
    loss = sum(z.square().mean() + p.mean() for z, p in zip(logits, probs))
    loss.backward()
    for nm, p in m.named_parameters():
        assert p.grad is not None, nm
        assert torch.isfinite(p.grad).all(), nm


# ------------------------------------------------------------------------------------------------------------------
# CUDA graph, level_cap, data parallel, launches
# ------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["unet_tl", "hrnet_tl"])
def test_channels_last_step_replays_from_a_cuda_graph(name):
    import rhseg_b200
    fx = Fixture(name)
    step = rhseg_b200.FusedHierStep(fx.tree, fx.level_weights)
    feats, hw, hb, fw, fb, target = _fx_leaves(fx, torch.float32, "cl")
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
                f.copy_(torch.randn(f.shape, generator=gen))
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
            assert a.stride() == b.stride()
            close(a, b, rtol=1e-6, what="graph grad %d/%d" % (it, i))
        for f, g in zip(feats, g_grads):
            assert is_cl(g)


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("name,cap", [("unet_tl", 0), ("hrnet_ext", 1)])
def test_level_cap_channels_last(name, cap, dtype):
    import rhseg_b200
    fx = Fixture(name)
    step = rhseg_b200.FusedHierStep(fx.tree, fx.level_weights)
    *leaves, target = _fx_leaves(fx, dtype, "cl")
    *ref_leaves, _ = _fx_leaves(fx, dtype, "nchw")
    out = step(*leaves, target, fx.out_size, level_cap=cap)
    out.loss.backward()
    ref = step(*ref_leaves, target, fx.out_size, level_cap=cap)
    ref.loss.backward()
    close(out.scalars, ref.scalars, what=f"{name} scalars")
    for L in range(fx.nL):
        a, r = leaves[0][L].grad, ref_leaves[0][L].grad
        if L > cap:
            assert (a is None and r is None) or (torch.count_nonzero(a) == 0 and torch.count_nonzero(r) == 0)
            continue
        assert is_cl(a)
        if dtype == BF:
            d = (a.double() - r.double()).abs()
            assert bool((d <= 2.0 ** -7 * r.double().abs() + 1e-5 * r.double().abs().max() + 1e-12).all())
        else:
            close(a, r, what=f"{name} dfeats{L}")


@gpu
@pytest.mark.parametrize("name,shards", [("unet_tl_odd_notooth", [slice(0, 1), slice(1, 3)]),
                                         ("hrnet_ext", [slice(0, 1), slice(1, 2)])])
def test_sharded_channels_last_step_equals_the_whole_batch(name, shards):
    import rhseg_b200
    fx = Fixture(name)
    world = len(shards)
    step = rhseg_b200.FusedHierStep(fx.tree, fx.level_weights)

    def leaves(sl=slice(None)):
        feats, hw, hb, fw, fb, target = _fx_leaves(fx, torch.float32, "cl")
        feats = [f.detach()[sl].contiguous(memory_format=CL).requires_grad_(True) for f in feats]
        return feats, hw, hb, fw, fb, target[sl].contiguous()

    feats, hw, hb, fw, fb, target = leaves()
    whole = step(feats, hw, hb, fw, fb, target, fx.out_size)
    whole.loss.backward()
    want_params = [p.grad.clone() for grp in (hw, hb, fw, fb) for p in grp]
    want_dfeats = [f.grad for f in feats]
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
                assert is_cl(f[L].grad)
                close(f[L].grad / world, want_dfeats[L][sl], what=f"{name} dfeats{L} shard {sl}")
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
    return sorted(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("name", ["unet_tl", "hrnet_tl"])
def test_channels_last_step_launches_no_copy(name, dtype):
    """The native channels-last step (forward + backward) launches as many kernels as the contiguous step, none of them
    a copy, a layout change or a conversion."""
    import rhseg_b200
    fx = Fixture(name)
    step = rhseg_b200.FusedHierStep(fx.tree, fx.level_weights)
    runs = {}
    for layout in ("nchw", "cl"):
        feats, hw, hb, fw, fb, target = _fx_leaves(fx, dtype, layout)
        leaves = feats + hw + hb + fw + fb

        def one_step():
            out = step(feats, hw, hb, fw, fb, target, fx.out_size)
            torch.autograd.grad(out.loss, leaves)

        one_step()
        runs[layout] = _kernel_names(one_step)
    assert len(runs["cl"]) == len(runs["nchw"]), (runs["cl"], runs["nchw"])
    # apart from the feature kernels, the same launches (the zero fills of the workspaces)
    other = lambda names: [n for n in names if "rhseg::" not in n]
    assert other(runs["cl"]) == other(runs["nchw"]), (other(runs["cl"]), other(runs["nchw"]))
    bad = [n for n in runs["cl"] if any(w in n.lower() for w in ("copy", "contiguous", "convert", "permute"))]
    assert not bad, bad
    assert any("nhwc" in n for n in runs["cl"]) and not any("nhwc" in n for n in runs["nchw"])


# ------------------------------------------------------------------------------------------------------------------
# without a GPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_channels_last_cpu_features_reach_the_device_check(dtype):
    import rhseg_b200
    from rhseg_b200 import native
    tree = rhseg_b200.ClassTree(TL)
    C = 16
    feats = [torch.zeros(1, C, 4, 4, dtype=dtype).contiguous(memory_format=CL) for _ in tree.head_channels]
    assert all(is_cl(f) for f in feats)
    hw = [torch.zeros(k, C, 1, 1) for k in tree.head_channels]
    hb = [torch.zeros(k) for k in tree.head_channels]
    fw = [torch.zeros(2 * C, tree.head_channels[0])]
    fb = [torch.zeros(2 * C)]
    with pytest.raises(native.NativeError, match="CUDA"):
        rhseg_b200.hier_head_forward(tree, feats, hw, hb, fw, fb)


def test_which_channels_last_tensors_are_read_in_place():
    from rhseg_b200 import head, native
    cl = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt).contiguous(memory_format=CL)
    assert head._nhwc_native(cl(2, 64, 5, 7))
    assert head._nhwc_native(cl(2, 720, 5, 7, dt=BF))
    assert not head._nhwc_native(torch.zeros(2, 64, 5, 7))           # contiguous: the NCHW path
    assert not head._nhwc_native(cl(2, 1, 5, 7))                     # C = 1: both layouts at once
    assert not head._nhwc_native(cl(2, 64, 1, 1))                    # 1x1 planes: both layouts at once
    assert not head._nhwc_native(cl(2, 18, 5, 7))                    # 72-byte pixels
    assert not head._nhwc_native(cl(2, 20, 5, 7, dt=BF))             # 40-byte pixels
    assert not head._nhwc_native(cl(2, 2048, 3, 3))                  # 8 KB pixels
    base = torch.zeros(2 * 64 * 5 * 7 + 4)
    assert not head._nhwc_native(base[1:1 + 2 * 64 * 35].view(2, 5, 7, 64).permute(0, 3, 1, 2))  # base off 16 bytes
    f, flags = head._feats_c([cl(2, 64, 5, 7), torch.zeros(2, 64, 5, 7), cl(2, 18, 5, 7)])
    assert flags == [native.FEATS_NHWC, 0, 0]
    assert is_cl(f[0]) and f[1].is_contiguous() and f[2].is_contiguous()
    _, flags = head._feats_c([cl(2, 64, 5, 7, dt=BF)])
    assert flags == [native.FEATS_NHWC | native.FEATS_BF16]


def test_feats_nhwc_flag_matches_the_header():
    from rhseg_b200 import native
    hdr = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "rhseg_b200.h")
    with open(hdr) as fh:
        txt = fh.read()
    assert int(re.search(r"#define RHSEG_FEATS_NHWC (0x[0-9a-fA-F]+)", txt).group(1), 16) == native.FEATS_NHWC
    assert native.FEATS_NHWC & native.FEATS_BF16 == 0
