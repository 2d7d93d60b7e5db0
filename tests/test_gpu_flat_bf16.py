"""bf16 logits (a flat head run under bf16 autocast) through FusedFlatStep and the drop-in losses.

Contract (DESIGN.md 3.10): with bf16 logits every result is what the fp32 path computes on logits.float() -- each logit
is widened to fp32 exactly when it is loaded, so the confusion matrix, the ratios and the train-path prediction are
bit-identical and the fp64 loss sums agree to rounding -- and dlogits is formed in fp32 and rounded to bf16 once, when
stored.  So the reference of every check here is the fp32 path on the upcast logits.  The dtype and flag checks at the
bottom run without a GPU."""
import os
import re

import numpy as np
import pytest
import torch

from helpers import GOLDEN, close
from oracle import hier_oracle as O
from test_gpu_bf16_features import TL, _small_hrnet_config, close_dfeats

DEV = "cuda"
BF = torch.bfloat16
gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNSUPPORTED = -2  # RHSEG_ERR_UNSUPPORTED


def _pair(z):
    """bf16 leaf and its exact fp32 upcast (another leaf)"""
    zb = z.detach().to(BF).to(DEV).requires_grad_(True)
    return zb, zb.detach().float().requires_grad_(True)


def _compare(out, ref, zb, zf, what):
    assert out.loss.dtype == torch.float32
    assert torch.equal(out.confusion[0], ref.confusion[0]), f"{what} confusion"
    assert torch.equal(out.ratios[0], ref.ratios[0]), f"{what} ratios"
    close(out.scalars, ref.scalars, what=f"{what} loss / CE / Dice")
    close(out.summary, ref.summary, what=f"{what} summary")
    close_dfeats(zb.grad, zf.grad, what=f"{what} dlogits")


def _run_pair(step, z, target, what):
    zb, zf = _pair(z)
    out = step(zb, target)
    out.loss.backward()
    ref = step(zf, target)
    ref.loss.backward()
    _compare(out, ref, zb, zf, what)
    return out, zb


# ------------------------------------------------------------------------------------------------------------------
# the flat7 reference fixture and the full-size flat7 workload
# ------------------------------------------------------------------------------------------------------------------
@gpu
def test_flat7_fixture_bf16_equals_fp32_on_upcast_logits():
    import rhseg_b200
    z = np.load(os.path.join(GOLDEN, "flat7.npz"))
    step = rhseg_b200.FusedFlatStep(7, [float(v) for v in z["weights"]])
    t = torch.from_numpy(z["target"]).float().to(DEV)
    _run_pair(step, torch.from_numpy(z["logits"]), t, "flat7")


@gpu
def test_flat7_full_size_bf16_against_fp32_and_the_fp64_oracle():
    import bench
    import rhseg_b200
    wl = bench.WORKLOADS["flat7_620_b4"]
    data = bench.synth_inputs(wl, wl["B"], seed=3, device="cpu")
    h = data["host"]
    target = h["target"]
    step = rhseg_b200.FusedFlatStep(wl["K"], data["weights"][0])
    out, zb = _run_pair(step, h["logits"], target.to(DEV), "flat7_620_b4")
    # fp64 oracle on the upcast logits (tests/test_gpu_fullsize.py does the same for fp32 logits)
    levels, parent_of, _, _ = O.hierarchy_tables(wl["tree"])
    zref = zb.detach().cpu().double().requires_grad_(True)
    loss_ref, _ = O.total_loss([zref], [target], data["weights"], None, levels, parent_of)
    loss_ref.backward()
    assert abs(out.loss.item() - loss_ref.item()) <= 1e-5 * abs(loss_ref.item()), (out.loss.item(), loss_ref.item())
    oh, et = O.predict_onehot_masked([zb.detach().float().cpu()], [target])
    assert torch.equal(out.confusion[0].cpu(), O.level_confusion(oh[0], et[0], wl["K"], False))
    close_dfeats(zb.grad, zref.grad, what="dlogits vs the fp64 oracle")


# ------------------------------------------------------------------------------------------------------------------
# every new kernel instance: K = 1..8, the pipelined and the fallback evaluation, both vector forms of the gradient
# and loss kernels
# ------------------------------------------------------------------------------------------------------------------
SHAPES = {            # (B, H, W): what rhseg_level_eval takes for them
    "pipe": (2, 48, 48),     # N % 16 == 0, B*N >= 4 * 1024: the bulk-copy pipeline
    "n16": (2, 44, 49),      # N % 4 == 0, N % 16 != 0: fallback, 4 pixels per thread (K <= 4)
    "odd": (2, 37, 41),      # N odd: fallback, one pixel per thread
    "small": (1, 32, 32),    # N % 16 == 0 but B*N below the pipeline's minimum
}


def _onehot_targets(B, K, H, W, gen, ignore=True):
    cls = torch.randint(0, K, (B, H, W), generator=gen)
    t = torch.nn.functional.one_hot(cls, K).permute(0, 3, 1, 2).float()
    if ignore:  # a few ignored pixels (-1 on every channel), as the dataset marks unlabeled ones
        t[:, :, :3, :5] = -1.0
    return t


def _bf16_at_offset(z, offset):
    """a view of a larger bf16 buffer whose base sits `offset` elements (2 bytes each) past a 16-byte boundary"""
    buf = torch.zeros(z.numel() + 16, dtype=BF, device=DEV)
    v = buf[offset:offset + z.numel()].view(z.shape)
    v.copy_(z)
    return v


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def _bf16_instances(names):
    """template argument lists of the launched bf16-logit instances, per kernel"""
    out = {}
    for n in names:
        m = re.search(r"(level_eval_pipe_kernel|level_eval_kernel|dz_fullres_fused_kernel|loss_stats_kernel|loss_bwd_kernel)<([^>]*)>",
                      n)
        if m and "unsigned short" in m.group(2):
            out.setdefault(m.group(1), set()).add(m.group(2).replace(" ", ""))
    return out


def _expected_instances():
    us = "unsignedshort"
    return {
        "level_eval_pipe_kernel": {"%d,0,%d,%s" % (k, k, us) for k in range(1, 9)},
        "level_eval_kernel": {"%d,4,2,256,-1,%s" % (k, us) for k in range(1, 5)}
        | {"%d,1,%d,256,-1,%s" % (k, 1 if k > 6 else 2, us) for k in range(1, 9)},
        "dz_fullres_fused_kernel": {"%d,%d,2,256,%s" % (k, v, us) for k in range(1, 9) for v in (1, 4)},
        "loss_stats_kernel": {"%d,%d,4,256,%s,%s" % (k, v, m, us) for k in range(1, 9) for v in (1, 4) for m in ("true", "false")},
        "loss_bwd_kernel": {"%d,%d,256,%s,%s" % (k, v, m, us) for k in range(1, 9) for v in (1, 4) for m in ("true", "false")},
    }


def _losses_pair(z, t, w, logits_input, what):
    """CrossEntropyLoss then SoftDiceLoss on the bf16 logits `z` (logits_input=False: on their softmax, rounded to bf16),
    one shared statistics pass, against the fp32 modules on the upcast tensor; the gradient is bf16 within the bound of
    the flat step."""
    import rhseg_b200
    from rhseg_b200.Metrics import losses
    K = z.shape[1]
    x = z if logits_input else torch.softmax(z.float(), dim=1).to(BF)
    zb = x.detach().requires_grad_(True)
    zf = zb.detach().float().requires_grad_(True)
    res = []
    for inp in (zb, zf):
        rhseg_b200.clear_memo()
        ce = losses.CrossEntropyLoss()(inp, t, class_weight=w, logits_input=logits_input)
        di = losses.SoftDiceLoss(num_classes=K)(inp, t, class_weight=w, logits_input=logits_input)
        assert ce.grad_fn is di.grad_fn, f"{what}: CE and Dice share one statistics node"
        (ce + di).backward()
        res.append((ce.detach(), di.detach()))
    close(res[0][0], res[1][0], what=f"{what} CE")
    close(res[0][1], res[1][1], what=f"{what} Dice")
    close_dfeats(zb.grad, zf.grad, what=f"{what} dz")


@gpu
def test_every_bf16_logit_instance_equals_fp32_on_upcast_logits():
    import rhseg_b200
    gen = torch.Generator().manual_seed(11)
    failures = []
    names = []

    def sweep():
        for K in range(1, 9):
            w = [0.5 + 0.1 * k for k in range(K)]
            step = rhseg_b200.FusedFlatStep(K, w)
            for shape, (B, H, W) in SHAPES.items():
                z = (torch.randn(B, K, H, W, generator=gen) * 3).to(BF).to(DEV)
                t = _onehot_targets(B, K, H, W, gen).to(DEV)
                wide = torch.cat([torch.zeros(B, 1, H, W, device=DEV), t, torch.zeros(B, 3, H, W, device=DEV)], 1)
                cases = [("fp32 targets", z, t), ("int8 targets", z, t.to(torch.int8)),
                         ("channel-slice targets", z, wide[:, 1:1 + K])]
                if shape == "pipe":
                    cases.append(("logits 2 bytes off 16", _bf16_at_offset(z, 1), t))
                for what, zz, tt in cases:
                    tag = "K=%d %s %s" % (K, shape, what)
                    try:
                        zb, zf = zz.detach().requires_grad_(True), zz.detach().float().requires_grad_(True)
                        if what.startswith("logits 2 bytes"):
                            assert zb.data_ptr() % 16 == 2
                        out = step(zb, tt)
                        out.loss.backward()
                        ref = step(zf, tt)
                        ref.loss.backward()
                        _compare(out, ref, zb, zf, tag)
                        for li in (True, False):
                            _losses_pair(zz, tt, w, li, "%s logits_input=%s" % (tag, li))
                    except AssertionError as e:
                        failures.append("%s: %s" % (tag, str(e).splitlines()[0]))

    names = _kernel_names(sweep)
    assert not failures, "\n".join(failures[:20])
    seen = _bf16_instances(names)
    for kern, want in _expected_instances().items():
        missing = want - seen.get(kern, set())
        assert not missing, "%s instances that never ran: %s" % (kern, sorted(missing))
    assert sum(len(v) for v in _expected_instances().values()) == 100


# ------------------------------------------------------------------------------------------------------------------
# drop-in losses on the reference fixture's logits
# ------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("logits_input", [True, False])
def test_dropin_losses_bf16_equal_fp32_on_upcast(logits_input):
    z = np.load(os.path.join(GOLDEN, "flat7.npz"))
    logits = torch.from_numpy(z["logits"]).to(BF).to(DEV)
    t = torch.from_numpy(z["target"]).float()
    wide = torch.cat([t, t[:, :2]], dim=1).to(DEV)  # the level's targets as a channel slice of a wider tensor
    _losses_pair(logits, wide[:, :7], [float(v) for v in z["weights"]], logits_input, "flat7 drop-in")


# ------------------------------------------------------------------------------------------------------------------
# flat models under autocast
# ------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("donor", ["unet", "hrnet"])
def test_flat_models_train_under_autocast(donor):
    import rhseg_b200
    from rhseg_b200.Metrics import losses
    from rhseg_b200.Models import models
    torch.manual_seed(7)
    if donor == "unet":
        m = models.UNet(size=32, n_channels=3, hierarchy=TL, model_type=0).to(DEV)
        x = torch.randn(2, 3, 32, 40, device=DEV)
    else:
        m = models.HighResolutionNet(_small_hrnet_config(), hierarchy=TL, model_type=0).to(DEV)
        x = torch.randn(2, 3, 36, 44, device=DEV)
    m.train()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        probs, z = m(x)
    # autocast runs the 1x1 conv in bf16 but keeps upsample_bilinear2d in fp32: UNet's flat logits (out_flat) are bf16,
    # HRNet's (classifier, then F.interpolate) come back fp32 and take the fp32 path
    assert probs == [] and z.dtype == (BF if donor == "unet" else torch.float32), z.dtype
    close_grad = (lambda a, r, what: close_dfeats(a, r.float(), what=what, roundings=2)) if z.dtype == BF else \
        (lambda a, r, what: close(a, r, what=what))
    K = z.shape[1]
    gen = torch.Generator().manual_seed(4)
    t = _onehot_targets(z.shape[0], K, z.shape[2], z.shape[3], gen).to(DEV)
    w = [1.0 + 0.1 * k for k in range(K)]
    step = rhseg_b200.FusedFlatStep(K, w)
    out, ref = step(z, t), step(z.float(), t)
    assert torch.equal(out.confusion[0], ref.confusion[0]) and torch.equal(out.ratios[0], ref.ratios[0])
    close(out.scalars, ref.scalars, what=f"{donor} step scalars")
    g, g_ref = torch.autograd.grad(out.loss, z, retain_graph=True)[0], torch.autograd.grad(ref.loss, z, retain_graph=True)[0]
    assert g.dtype == z.dtype
    close_grad(g, g_ref, f"{donor} step dlogits")
    rhseg_b200.clear_memo()
    ce = losses.CrossEntropyLoss()(z, t, class_weight=w, logits_input=True)
    di = losses.SoftDiceLoss(num_classes=K)(z, t, class_weight=w, logits_input=True)
    rhseg_b200.clear_memo()
    ce_f = losses.CrossEntropyLoss()(z.float(), t, class_weight=w, logits_input=True)
    di_f = losses.SoftDiceLoss(num_classes=K)(z.float(), t, class_weight=w, logits_input=True)
    close(ce, ce_f, what=f"{donor} CE")
    close(di, di_f, what=f"{donor} Dice")
    gl = torch.autograd.grad(ce + di, z, retain_graph=True)[0]
    gl_ref = torch.autograd.grad(ce_f + di_f, z, retain_graph=True)[0]
    close_grad(gl, gl_ref, f"{donor} drop-in dlogits")
    (out.loss + ce + di).backward()
    for nm, p in m.named_parameters():
        if p.requires_grad:
            assert p.grad is not None, nm
            assert torch.isfinite(p.grad).all(), nm


# ------------------------------------------------------------------------------------------------------------------
# no hidden cast, CUDA graphs
# ------------------------------------------------------------------------------------------------------------------
@gpu
def test_bf16_flat_step_launches_what_the_fp32_step_launches():
    import rhseg_b200
    step = rhseg_b200.FusedFlatStep(7, [1.0] * 7)
    gen = torch.Generator().manual_seed(2)
    z32 = torch.randn(2, 7, 64, 64, generator=gen).to(DEV)
    t = _onehot_targets(2, 7, 64, 64, gen).to(DEV)
    runs = {}
    for dt in (torch.float32, BF):
        z = z32.to(dt).requires_grad_(True)

        def one_step():
            out = step(z, t)
            g = torch.autograd.grad(out.loss, z)[0]
            assert g.dtype == dt

        one_step()  # warm: tables, weights
        runs[dt] = sorted(n.split("<")[0] for n in _kernel_names(one_step))
    assert runs[BF] == runs[torch.float32], (runs[BF], runs[torch.float32])
    assert not any("copy" in n.lower() or "convert" in n.lower() for n in runs[BF]), runs[BF]


@gpu
def test_bf16_flat_step_replays_from_a_cuda_graph():
    import rhseg_b200
    step = rhseg_b200.FusedFlatStep(7, [0.5 + 0.2 * k for k in range(7)])
    gen = torch.Generator().manual_seed(5)
    z = (torch.randn(4, 7, 96, 96, generator=gen) * 2).to(BF).to(DEV).requires_grad_(True)
    t = _onehot_targets(4, 7, 96, 96, gen).to(DEV)
    one = torch.ones((), device=DEV)

    def run():
        out = step(z, t)
        return out, torch.autograd.grad(out.loss, z, grad_outputs=one)[0]

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            run()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_out, g_grad = run()
    for it in range(2):
        with torch.no_grad():
            z.copy_((torch.randn(z.shape, generator=gen) * 2).to(BF))
        graph.replay()
        torch.cuda.synchronize()
        got = (g_out.scalars.clone(), g_out.confusion[0].clone(), g_out.ratios[0].clone(), g_grad.clone())
        e_out, e_grad = run()
        torch.cuda.synchronize()
        close(got[0], e_out.scalars, what="graph scalars %d" % it)
        assert torch.equal(got[1], e_out.confusion[0]) and torch.equal(got[2], e_out.ratios[0])
        assert got[3].dtype == BF
        # the order of fp64 atomics may move an fp32 value across a bf16 rounding boundary
        close_dfeats(got[3], e_grad.float(), what="graph dlogits %d" % it, roundings=2)


# ------------------------------------------------------------------------------------------------------------------
# C-ABI: flagged calls that reach an instance without a bf16 form
# ------------------------------------------------------------------------------------------------------------------
@gpu
def test_c_abi_rejects_bf16_logits_where_there_is_no_bf16_instance():
    import rhseg_b200
    from rhseg_b200 import native
    from rhseg_b200.native import ptr
    lib = native.lib()
    B, K, N = 1, 4, 256
    z = torch.zeros(B, K, N, dtype=BF, device=DEV)
    t = torch.zeros(B, K, N, device=DEV)
    ws = torch.zeros(B * K * native.NSTAT + native.MAX_K + (K + 1) ** 2, dtype=torch.float64, device=DEV)
    idx = torch.zeros(B, N, dtype=torch.uint8, device=DEV)
    table = rhseg_b200.ClassTree(TL).device_tables(DEV)[1]
    st = native.stream_of(z)
    F = native.LOGITS_BF16
    ev = lambda child, pt, prev, out: lib.rhseg_level_eval(ptr(z), ptr(t), K * N, N, pt, K * N, N, prev, ptr(table), B, K, N,
                                                           child, ptr(ws), out, F, st)
    for what, rc in [("child level", ev(1, None, None, None)),
                     ("child level with a group hint", ev(1 | (4 << 8), None, None, None)),
                     ("parent targets", ev(0, ptr(t), None, None)),
                     ("prev_idx", ev(0, None, ptr(idx), None)),
                     ("idx_out", ev(0, None, None, ptr(idx)))]:
        assert rc == UNSUPPORTED, (what, rc)
    coef = torch.zeros(B * K * 3, device=DEV)
    dz = torch.empty_like(z)
    prev = torch.zeros(B, 3, N, device=DEV)
    for mode in (native.ACT_SIGMOID, native.ACT_GROUPED, native.ACT_GROUPED | (4 << 8)):
        rc = lib.rhseg_head_dz_fullres_fused(ptr(z), ptr(t), K * N, N, ptr(coef), None, None, ptr(prev), ptr(table), None,
                                             1.0 / N, None, 0, B, K, 3, N, mode | F, ptr(dz), None, st)
        assert rc == UNSUPPORTED, (mode, rc)
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------------------------
# dtype validation and the flag value (no GPU needed)
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float16, torch.float64])
def test_other_logit_dtypes_are_refused(dtype):
    import rhseg_b200
    from rhseg_b200 import native
    from rhseg_b200.Metrics import losses
    z = torch.zeros(1, 7, 4, 4, dtype=dtype)
    t = torch.zeros(1, 7, 4, 4)
    with pytest.raises(native.NativeError, match="bfloat16"):
        rhseg_b200.FusedFlatStep(7, [1.0] * 7)(z, t)
    for li in (True, False):
        with pytest.raises(native.NativeError, match="bfloat16"):
            losses.CrossEntropyLoss()(z, t, class_weight=[1.0] * 7, logits_input=li)


def test_bf16_cpu_logits_reach_the_device_check():
    """bf16 passes the dtype check and fails only because there is no CPU path"""
    from rhseg_b200 import native
    from rhseg_b200.Metrics import losses
    with pytest.raises(native.NativeError, match="CUDA"):
        losses.CrossEntropyLoss()(torch.zeros(1, 7, 4, 4, dtype=BF), torch.zeros(1, 7, 4, 4), class_weight=[1.0] * 7,
                                  logits_input=True)


def _header_define(name):
    with open(os.path.join(ROOT, "include", "rhseg_b200.h")) as f:
        m = re.search(r"^#define %s\s+(\S+)" % name, f.read(), flags=re.M)
    return int(m.group(1), 0)


def test_logits_flag_matches_the_header_and_shares_no_bit():
    from rhseg_b200 import native
    flag = native.LOGITS_BF16
    assert flag == _header_define("RHSEG_LOGITS_BF16")
    assert flag & (flag - 1) == 0, "one bit"
    taken = [_header_define("RHSEG_EVAL_PREZEROED"), native.ACT_SIGMOID | native.ACT_GROUPED | native.ACT_ZEROS,
             255 << 8, 1]  # RHSEG_GROUP_HINT(255); logits_input 0 / 1
    for bits in taken:
        assert flag & bits == 0, hex(bits)
