"""Fused validation (FusedHierStep.validate, rhseg_level_eval_composed): the numbers of the reference's test() pass
(train.py:324-339) in one forward without autograd and without a host sync.

The evaluation differs from the training step's (DESIGN.md 3.9): the confusion matrix is ProcessClasses over the composed
probabilities against the raw ternary targets, and the consistency term is taken on the real probabilities.  CE and Dice
are the step's.  References: the fixtures' recorded CE / Dice / `consistency_eval`, the oracle's confusion and ratios,
and (C-ABI sweep) the single-purpose kernels rhseg_loss_stats, rhseg_confusion_matrix and rhseg_consistency_sums on the
same tensors.  The checks at the bottom run without a GPU."""
import ctypes
import math
import os
import re

import pytest
import torch

from helpers import HIER_CASES, Fixture, close
from oracle import hier_oracle as O

DEV = "cuda"
BF = torch.bfloat16
gpu = pytest.mark.gpu


def _leaves(fx, requires_grad=False, sl=slice(None), dtype=torch.float32, layout=None):
    mk = lambda ts: [t.to(DEV).requires_grad_(requires_grad) for t in ts]
    feats = []
    for t in fx.per_level("feats"):
        t = t[sl].to(dtype).to(DEV)
        t = t.contiguous(memory_format=torch.channels_last) if layout == "cl" else t.contiguous()
        feats.append(t.requires_grad_(requires_grad))
    hw, hb = mk(fx.per_level("head_w")), mk(fx.per_level("head_b"))
    fw, fb = mk(fx.per_level("film_w", n=fx.nL - 1)), mk(fx.per_level("film_b", n=fx.nL - 1))
    target = torch.cat(fx.per_level("target"), dim=1)[sl].contiguous().to(DEV)
    return feats, hw, hb, fw, fb, target


def _step(fx):
    import rhseg_b200
    return rhseg_b200.FusedHierStep(fx.tree, fx.level_weights)


# ---------------------------------------------------------------------------------------------------------------------
# reference parity
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", HIER_CASES)
def test_validate_matches_reference(name):
    import rhseg_b200
    fx = Fixture(name)
    step = _step(fx)
    feats, hw, hb, fw, fb, target = _leaves(fx)
    # the wide target sits inside a larger buffer so that level slices are strided views
    wide = torch.zeros(target.shape[0], target.shape[1] + 3, *target.shape[2:], device=DEV)
    wide[:, 1:1 + target.shape[1]] = target
    out = step.validate(feats, hw, hb, fw, fb, wide[:, 1:1 + target.shape[1]], fx.out_size, keep_outputs=True)
    want_total = fx.f("consistency_eval")
    for L in range(fx.nL):
        assert abs(out.level_ce[L].item() - fx.f(f"ce{L}")) <= 1e-5 * max(1.0, abs(fx.f(f"ce{L}")))
        want_total += fx.f(f"ce{L}")
        if math.isnan(fx.f(f"dice{L}")):
            assert out.level_dice[L].item() == 0.0 and out.scalars[4 + 4 * L].item() == 0.0
        else:
            assert abs(out.level_dice[L].item() - fx.f(f"dice{L}")) <= 1e-5
            want_total += fx.f(f"dice{L}")
    assert abs(out.consistency.item() - fx.f("consistency_eval")) <= 1e-7
    assert abs(out.loss.item() - want_total) <= 1e-5 * abs(want_total), (out.loss.item(), want_total)
    tree = rhseg_b200.ClassTree(fx.tree)
    with torch.no_grad():
        probs, _ = rhseg_b200.hier_head_forward(tree, feats, hw, hb, fw, fb, fx.out_size)
    for L in range(fx.nL):
        assert torch.equal(out.probs[L], probs[L]), f"{name} probs{L}"
        want = O.level_confusion(probs[L].cpu(), fx.t(f"target{L}"), tree.head_channels[L], L != 0)
        assert torch.equal(out.confusion[L].cpu(), want), f"{name} confusion{L}"
        r = O.ratios_from_confusion(want)
        for row, key in enumerate(("dice", "iou", "accuracy", "precision", "recall")):
            assert torch.equal(out.ratios[L][row].cpu(), r[key]), (name, L, key)


@gpu
@pytest.mark.parametrize("name", ["unet_ext", "hrnet_ext"])
def test_validate_is_not_the_training_evaluation(name):
    """On a level with two parent groups the train-path prediction argmax(softmax z) and ProcessClasses(P) disagree on
    some pixels; validate reports the latter, the training step the former."""
    import rhseg_b200
    fx = Fixture(name)
    tree = rhseg_b200.ClassTree(fx.tree)
    L = next(L for L in range(1, fx.nL) if tree.group_count(L) >= 2)
    z, P = fx.t(f"logits{L}"), fx.t(f"probs{L}")
    assert bool((z.argmax(1) != P.argmax(1)).any()), "fixture has no pixel that tells the two predictions apart"
    step = _step(fx)
    leaves = _leaves(fx)
    val = step.validate(*leaves, fx.out_size)
    with torch.no_grad():
        train = step(*leaves, fx.out_size)
    assert not torch.equal(val.confusion[L], train.confusion[L])
    assert abs(val.consistency.item() - train.consistency.item()) > 1e-3
    close(val.scalars[2:], train.scalars[2:], what="per-level CE / Dice")  # the same statistics


# ---------------------------------------------------------------------------------------------------------------------
# C-ABI sweep against the single-purpose kernels
# ---------------------------------------------------------------------------------------------------------------------
def _layouts(K):
    """(name, parent channel per child channel, K_prev, group hint) of the child levels the sweep runs at width K"""
    out = [("one_group", [0] * K, 2, K)]  # hint == K: the compile-time layout
    if K >= 3:
        out.append(("ragged", [0] + [1] * (K - 1), 3, 0))  # groups of 1 and K-1 plus a parent without children
    else:
        out.append(("no_hint", [1] * K, 2, 0))
    if K == 4:
        out.append(("two_pairs", [0, 0, 2, 2], 3, 2))
    return out


def _run_sweep_case(K, kind, layout, B, H, W, t_pad, gen):
    """One call of rhseg_level_eval_composed against rhseg_loss_stats / rhseg_confusion_matrix / rhseg_consistency_sums.
    kind: 0 root, 1 child, 2 child + consistency.  t_pad: extra elements per target plane (strided, unaligned)."""
    from rhseg_b200 import native
    N = H * W
    name, parent_ch, K_prev, hint = layout if kind else ("root", [-1] * K, 0, 0)
    table = torch.tensor(native.compile_level_table(parent_ch, K_prev), dtype=torch.int32, device=DEV)
    logits = (torch.randn(B, K, N, generator=gen) * 3).to(DEV)
    probs = torch.rand(B, K, N, generator=gen)
    probs[:, :, : N // 7] = 0.0                     # "nothing positive" pixels
    probs[:, :, N // 7: N // 5] = 0.25              # ties: first maximum wins
    probs = probs.to(DEV)
    tern = torch.randint(-1, 2, (B, K, N), generator=gen).float()
    tbuf = torch.zeros(B, K + 1, N + t_pad)
    tbuf[:, 1:, :N] = tern
    tbuf = tbuf.to(DEV)
    targets = tbuf[:, 1:, :N]
    t_bs, t_cs = tbuf.stride(0), tbuf.stride(1)
    prev = None
    if kind == 2:
        # the previous level's probabilities: each parent channel close to the sum of its children (as composed
        # probabilities are), the rest random, so that a wrong parent or group shows as an O(1) error
        prev = torch.rand(B, K_prev, N, generator=gen)
        pc = torch.tensor(parent_ch)
        for p in sorted(set(parent_ch)):
            prev[:, p] = probs.cpu()[:, pc == p].sum(1) + (torch.rand(B, N, generator=gen) - 0.5) * 2e-3
        prev = prev.to(DEV)
    nc = K + 1 if kind else K
    words = torch.full((B * K * native.NSTAT + native.MAX_K + nc * nc,), 7.0, dtype=torch.float64, device=DEV)
    st = native.stream_of(logits)
    native.call("rhseg_level_eval_composed", logits.data_ptr(), probs.data_ptr(), native.ptr(prev), targets.data_ptr(),
                t_bs, t_cs, table.data_ptr(), B, K, K_prev, N, (1 if kind else 0) | (hint << 8), words.data_ptr(), 0, st)
    stats = torch.empty(B * K * native.NSTAT, dtype=torch.float64, device=DEV)
    native.call("rhseg_loss_stats", logits.data_ptr(), targets.data_ptr(), t_bs, t_cs, B, K, N, 1, stats.data_ptr(), st)
    conf = torch.empty(nc * nc, dtype=torch.int64, device=DEV)
    native.call("rhseg_confusion_matrix", probs.data_ptr(), K * N, N, targets.data_ptr(), t_bs, t_cs, B, K, N,
                1 if kind else 0, conf.data_ptr(), st)
    torch.cuda.synchronize()
    tag = "K=%d kind=%d %s %dx%dx%d pad=%d" % (K, kind, name, B, H, W, t_pad)
    o = B * K * native.NSTAT
    close(words[:o], stats, what=tag + " stats")
    assert torch.equal(words[o + native.MAX_K:].view(torch.int64), conf), tag + " confusion"
    got_cons = words[o:o + native.MAX_K]
    if kind == 2:
        sums = torch.empty(native.MAX_K, dtype=torch.float64, device=DEV)
        native.call("rhseg_consistency_sums", probs.data_ptr(), prev.data_ptr(), table.data_ptr(), B, K, K_prev, N,
                    sums.data_ptr(), st)
        torch.cuda.synchronize()
        n_g = len(set(parent_ch))
        close(got_cons[:n_g], sums[:n_g], what=tag + " consistency sums")
        assert bool((got_cons[n_g:] == 0).all()) and sums[:n_g].min().item() > 0.0
    else:
        assert bool((got_cons == 0).all()), tag + " consistency slots"


SWEEP_SHAPES = [(2, 48, 64, 0),    # pipeline: aligned planes, N % 4 == 0, strided target slices
                (3, 17, 23, 0),    # odd planes: one-pixel-per-thread kernel
                (2, 10, 30, 0),    # N % 16 != 0, N % 4 == 0: pipeline, a stage ends mid-way
                (2, 48, 64, 1)]    # target planes off the 16-byte grid: one-pixel-per-thread kernel


def _kernel_names(prof):
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


def _instances(names, kernel):
    out = set()
    for n in names:
        m = re.search(kernel + r"<([0-9, ]+)>", n)
        if m:
            out.add(tuple(int(x) for x in m.group(1).split(",")))
    return out


@gpu
@pytest.mark.parametrize("K", range(1, 9))
def test_level_eval_composed_sweep(K):
    gen = torch.Generator().manual_seed(100 + K)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for shape in SWEEP_SHAPES:
            _run_sweep_case(K, 0, None, *shape, gen)
            for layout in _layouts(K):
                for kind in (1, 2):
                    _run_sweep_case(K, kind, layout, *shape, gen)
        torch.cuda.synchronize()
    names = _kernel_names(prof)
    want_pipe = {(K, 0, K), (K, 1, K), (K, 2, K), (K, 1, 0), (K, 2, 0)} | ({(4, 1, 2), (4, 2, 2)} if K == 4 else set())
    assert _instances(names, "level_val_pipe_kernel") == want_pipe
    assert _instances(names, "level_val_kernel") == {(K, 0), (K, 1), (K, 2)}


def _run_band_case(K, layout, B, C, Hf, Wf, H, W, gen):
    """rhseg_head_level_fwd_eval with RHSEG_EVAL_COMPOSED against rhseg_level_eval_composed on the logits and
    probabilities the same call wrote.  layout None: the sigmoid root level."""
    from rhseg_b200 import native
    N = H * W
    if layout is None:
        name, parent_ch, K_prev, hint, act = "root", [-1] * K, 0, 0, native.ACT_SIGMOID
    else:
        (name, parent_ch, K_prev, hint), act = layout, native.ACT_GROUPED
    table = torch.tensor(native.compile_level_table(parent_ch, K_prev), dtype=torch.int32, device=DEV)
    feats = torch.randn(B, C, Hf, Wf, generator=gen).to(DEV)
    eff_w = (torch.randn(K, C, generator=gen) * 0.5).to(DEV)
    eff_b = (torch.randn(K, generator=gen) * 0.1).to(DEV)
    prev = torch.rand(B, K_prev, H, W, generator=gen).to(DEV) if K_prev else None
    tern = torch.randint(-1, 2, (B, K + 1, H, W), generator=gen).float().to(DEV)
    targets = tern[:, 1:]
    t_bs, t_cs = tern.stride(0), tern.stride(1)
    z_lo = torch.zeros(B, K, Hf, Wf, device=DEV)
    logits = torch.empty(B, K, H, W, device=DEV)
    probs = torch.empty(B, K, H, W, device=DEV)
    psum = torch.zeros(B, K, dtype=torch.float64, device=DEV)
    nc = K + 1 if layout else K
    n_words = B * K * native.NSTAT + native.MAX_K + nc * nc
    words = torch.full((n_words,), 7.0, dtype=torch.float64, device=DEV)
    junk = torch.full((B, H, W), 255, dtype=torch.uint8, device=DEV)  # ignored in the composed mode
    st = native.stream_of(feats)
    native.call("rhseg_head_level_fwd_eval", feats.data_ptr(), eff_w.data_ptr(), eff_b.data_ptr(), native.ptr(prev),
                table.data_ptr(), B, C, Hf, Wf, H, W, K, K_prev, act | (hint << 8), z_lo.data_ptr(), logits.data_ptr(),
                probs.data_ptr(), psum.data_ptr(), targets.data_ptr(), t_bs, t_cs, targets.data_ptr(), t_bs, t_cs,
                junk.data_ptr(), words.data_ptr(), junk.data_ptr(), native.EVAL_COMPOSED | 2 | 4, st)
    ref = torch.zeros(n_words, dtype=torch.float64, device=DEV)
    native.call("rhseg_level_eval_composed", logits.data_ptr(), probs.data_ptr(), native.ptr(prev), targets.data_ptr(),
                t_bs, t_cs, table.data_ptr(), B, K, K_prev, N, (1 if layout else 0) | (hint << 8), ref.data_ptr(), 1, st)
    torch.cuda.synchronize()
    tag = "band K=%d %s %dx%d -> %dx%d" % (K, name, Hf, Wf, H, W)
    o = B * K * native.NSTAT
    close(words[:o], ref[:o], what=tag + " stats")
    # the band kernel composes P from the same parent plane it compares with, so the sums are rounding residues here;
    # the stand-alone sweep above checks the parent mapping with sums of O(1e-3) per pixel
    close(words[o:o + native.MAX_K], ref[o:o + native.MAX_K], what=tag + " consistency sums")
    assert torch.equal(words[o + native.MAX_K:].view(torch.int64), ref[o + native.MAX_K:].view(torch.int64)), tag + " confusion"
    assert bool((junk == 255).all()), tag + " index map written"


@gpu
@pytest.mark.parametrize("K", range(1, 9))
def test_band_forward_composed_eval_sweep(K):
    """The validation evaluation inside the HRNet band forward equals the stand-alone kernel's on the same outputs, for
    every band instance it is built for (4 pixels per thread at scale 4, 2 at scale 2 for K <= 4; group layouts fixed at
    compile time or, up to K = 6, read from the table); the other shapes take the generic forward + the stand-alone
    evaluation, with the same results."""
    gen = torch.Generator().manual_seed(300 + K)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for (Hf, H) in ((12, 48), (12, 24)):
            _run_band_case(K, None, 2, 16, Hf, Hf, H, H, gen)
            for layout in _layouts(K):
                _run_band_case(K, layout, 2, 16, Hf, Hf, H, H, gen)
        torch.cuda.synchronize()
    got = {t for t in _instances(_kernel_names(prof), "upsample_band_kernel") if t[3] == 3}
    want = set()
    for vec in ([4, 2] if K <= 4 else [4]):
        want |= {(K, vec, 0, 3, K), (K, vec, 1, 3, K)}
        if K <= 6:
            want.add((K, vec, 1, 3, 0))
        if K == 4:
            want.add((K, vec, 1, 3, 2))
    assert got == want


@gpu
def test_level_eval_composed_argument_errors():
    from rhseg_b200 import native
    x = torch.zeros(2, 4, 64, device=DEV)
    words = torch.zeros(64, dtype=torch.float64, device=DEV)
    table = torch.zeros(native.TABLE_INTS, dtype=torch.int32, device=DEV)
    lib = native.lib()
    p = x.data_ptr()
    assert lib.rhseg_level_eval_composed(None, p, None, p, 256, 64, None, 2, 4, 0, 64, 0, words.data_ptr(), 0, None) == -1
    assert lib.rhseg_level_eval_composed(p, p, None, p, 256, 64, None, 2, 4, 0, 64, 1, words.data_ptr(), 0, None) == -1  # child, no table
    assert lib.rhseg_level_eval_composed(p, p, p, p, 256, 64, table.data_ptr(), 2, 4, 0, 64, 1, words.data_ptr(), 0, None) == -1  # K_prev
    assert lib.rhseg_level_eval_composed(p, p, None, p, 256, 64, None, 2, 9, 0, 64, 0, words.data_ptr(), 0, None) == -2
    assert lib.rhseg_level_eval_composed(p, p, None, p, 256, 64, None, 0, 4, 0, 64, 0, words.data_ptr(), 0, None) == -1


# ---------------------------------------------------------------------------------------------------------------------
# step-level properties
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["unet_tl", "hrnet_ext"])
def test_validate_feature_dtypes_and_layouts(name):
    """bf16 features give what the upcast fp32 features give, bit for bit (DESIGN.md 3.8: each bf16 value converts to
    fp32 exactly).  Channels-last features: confusion exact; at feature resolution (UNet) the logits and probabilities
    are bit-identical, so the scalars are too; upsampled heads agree to rounding."""
    fx = Fixture(name)
    step = _step(fx)
    upcast = _leaves(fx, dtype=BF)
    upcast = ([f.float() for f in upcast[0]],) + upcast[1:]
    ref = step.validate(*upcast, fx.out_size)
    bf = step.validate(*_leaves(fx, dtype=BF), fx.out_size)
    assert torch.equal(bf.scalars, ref.scalars)
    for a, b in zip(bf.confusion, ref.confusion):
        assert torch.equal(a, b)
    for dtype in (torch.float32, BF):
        nchw = step.validate(*_leaves(fx, dtype=dtype), fx.out_size)
        cl_leaves = _leaves(fx, dtype=dtype, layout="cl")
        assert not cl_leaves[0][0].is_contiguous()
        cl = step.validate(*cl_leaves, fx.out_size)
        for a, b in zip(cl.confusion, nchw.confusion):
            assert torch.equal(a, b)
        if fx.out_size is None:
            assert torch.equal(cl.scalars, nchw.scalars)
        else:
            close(cl.scalars, nchw.scalars, what=f"{name} channels-last scalars")


@gpu
def test_validate_records_no_graph_no_sync_no_extra_memory():
    fx = Fixture("hrnet_ext")
    step = _step(fx)
    leaves = _leaves(fx, requires_grad=True)
    with torch.enable_grad():
        step.validate(*leaves, fx.out_size)  # warm-up: device tables, weights
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            out = step.validate(*leaves, fx.out_size)
        finally:
            torch.cuda.set_sync_debug_mode(0)
    assert out.loss.grad_fn is None and not out.loss.requires_grad
    assert out.probs == [None] * fx.nL and out.logits == [None] * fx.nL
    del out

    def peak(fn):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()  # releases blocks still waiting for a side-stream event, so they do not offset the peak
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        r = fn()
        torch.cuda.synchronize()
        p = torch.cuda.max_memory_allocated() - base
        del r
        return p

    def train_no_grad():
        with torch.no_grad():
            return step(*leaves, fx.out_size)

    p_step = peak(train_no_grad)
    with torch.enable_grad():
        p_val = peak(lambda: step.validate(*leaves, fx.out_size))
    assert p_val <= p_step, (p_val, p_step)


@gpu
def test_validate_replays_from_a_cuda_graph():
    fx = Fixture("hrnet_ext")
    step = _step(fx)
    feats, hw, hb, fw, fb, target = _leaves(fx)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step.validate(feats, hw, hb, fw, fb, target, fx.out_size)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_out = step.validate(feats, hw, hb, fw, fb, target, fx.out_size)
    gen = torch.Generator().manual_seed(7)
    for it in range(2):
        for f in feats:
            f.copy_(torch.randn(f.shape, generator=gen))
        graph.replay()
        torch.cuda.synchronize()
        got = (g_out.scalars.clone(), [c.clone() for c in g_out.confusion], g_out.summary.clone())
        e_out = step.validate(feats, hw, hb, fw, fb, target, fx.out_size)
        torch.cuda.synchronize()
        close(got[0], e_out.scalars, rtol=1e-6, what="graph scalars %d" % it)  # only the order of fp64 atomics differs
        for a, b in zip(got[1], e_out.confusion):
            assert torch.equal(a, b)


@gpu
@pytest.mark.parametrize("cap", [0, 1])
def test_validate_level_cap(cap):
    fx = Fixture("unet_ext")
    step = _step(fx)
    leaves = _leaves(fx)
    full = step.validate(*leaves, fx.out_size)
    capped = step.validate(*leaves, fx.out_size, level_cap=cap)
    want = capped.consistency.item() + sum(capped.level_ce[L].item() + capped.level_dice[L].item() for L in range(cap + 1))
    assert abs(capped.loss.item() - want) <= 1e-6 * abs(want)
    close(capped.scalars[1:], full.scalars[1:], rtol=1e-6, what="every level is still reported")
    for a, b in zip(capped.confusion, full.confusion):
        assert torch.equal(a, b)


@gpu
@pytest.mark.parametrize("name", ["unet_tl_odd_notooth", "hrnet_ext"])
def test_validate_summary_is_additive(name):
    """The summary of a batch is the sum of its halves' summaries (confusion exactly; the loss sums to the rounding of
    the fp32 per-CTA partials, whose split over CTAs depends on the batch), and a data-parallel validate with a
    stand-in all-reduce reports the global numbers of the whole batch."""
    from rhseg_b200 import dist as rdist
    fx = Fixture(name)
    step = _step(fx)
    whole = step.validate(*_leaves(fx), fx.out_size)
    B = fx.B
    halves = [slice(0, B // 2), slice(B // 2, B)]
    parts = [step.validate(*_leaves(fx, sl=sl), fx.out_size).summary.clone() for sl in halves]
    gsum = parts[0] + parts[1]
    n_scal = 2 + 4 * fx.nL
    assert torch.equal(gsum[n_scal:], whole.summary[n_scal:])  # confusion counts
    close(gsum[:n_scal], whole.summary[:n_scal], rtol=1e-6, what="additive loss sums")
    shapes = [tuple(c.shape) for c in whole.confusion]
    glob = rdist.unpack_global(gsum, fx.nL, shapes)
    assert abs(glob["total"].item() - whole.loss.item()) <= 1e-6 * abs(whole.loss.item())
    step.data_parallel(lambda s: gsum.clone(), len(halves))
    for sl in halves:
        out = step.validate(*_leaves(fx, sl=sl), fx.out_size)
        assert torch.equal(out.global_summary, gsum)
        g = rdist.unpack_global(out.global_summary, fx.nL, shapes)
        for L in range(fx.nL):
            assert torch.equal(g["confusion"][L], whole.confusion[L])


@gpu
def test_validate_int8_targets():
    fx = Fixture("hrnet_ext")
    step = _step(fx)
    feats, hw, hb, fw, fb, target = _leaves(fx)
    a = step.validate(feats, hw, hb, fw, fb, target, fx.out_size)
    b = step.validate(feats, hw, hb, fw, fb, target.to(torch.int8), fx.out_size)
    close(a.scalars, b.scalars, rtol=1e-6, what="int8 targets")
    for x, y in zip(a.confusion, b.confusion):
        assert torch.equal(x, y)


# ---------------------------------------------------------------------------------------------------------------------
# without a GPU
# ---------------------------------------------------------------------------------------------------------------------
def test_validate_argument_errors():
    import rhseg_b200
    from rhseg_b200 import native
    fx = Fixture("unet_tl")
    step = rhseg_b200.FusedHierStep(fx.tree, fx.level_weights)
    feats = fx.per_level("feats")
    hw, hb = fx.per_level("head_w"), fx.per_level("head_b")
    fw, fb = fx.per_level("film_w", n=fx.nL - 1), fx.per_level("film_b", n=fx.nL - 1)
    target = torch.cat(fx.per_level("target"), dim=1)
    with pytest.raises(native.NativeError):
        step.validate(feats[:-1], hw, hb, fw, fb, target)
    with pytest.raises(native.NativeError):  # no CPU fallback
        step.validate(feats, hw, hb, fw, fb, target)


def test_eval_composed_flag_matches_the_header():
    from rhseg_b200 import native
    hdr = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "rhseg_b200.h")
    with open(hdr) as fh:
        txt = fh.read()
    assert int(re.search(r"#define RHSEG_EVAL_COMPOSED (0x[0-9a-fA-F]+)", txt).group(1), 16) == native.EVAL_COMPOSED
    taken = 1 | 2 | 4 | native.FEATS_BF16 | native.FEATS_NHWC  # the other bits of rhseg_head_level_fwd_eval's flags
    assert native.EVAL_COMPOSED & taken == 0


def test_level_eval_composed_binding_matches_the_header():
    from rhseg_b200 import native
    hdr = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "rhseg_b200.h")
    with open(hdr) as fh:
        txt = fh.read()
    proto = re.search(r"int rhseg_level_eval_composed\(([^)]*)\);", txt).group(1)
    kinds = []
    for arg in proto.split(","):
        arg = arg.strip()
        kinds.append(ctypes.c_void_p if "*" in arg else ctypes.c_long if arg.startswith("long") else ctypes.c_int)
    assert native.SIGNATURES["rhseg_level_eval_composed"] == kinds
