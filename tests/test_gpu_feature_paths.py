"""Every feature path of the head -- fp32 / bf16 donor features, contiguous (NCHW) / channels-last (NHWC) -- against a
plain float64 restatement of the same operation, never against another device path.

  part 0  the fp64 reference (level forward, conv backward) and a CPU check that it reproduces the oracle's head
  part 1  every kernel instance through the C-ABI: K = 1..8 x {sigmoid, grouped, zeros} x both tile shapes, the
          low-resolution conv, the conv backward with per-sample / shared weights and without dfeats; a profiler
          check that every NHWC instance (128) and every targeted NCHW instance ran
  part 2  the persistent-grid paths small fixtures never reach (sample change inside a CTA, low-res tiles split
          between CTAs, the backward's 64-unit flush) and the channel counts at the edges of the NHWC contract
  part 3  the full-size workloads through FusedHierStep in all four dtype x layout combinations

Inputs are bf16-representable in every dtype, so one fp64 reference serves fp32 and bf16 alike.  Tolerances:
helpers.close's bound at 1e-5 (|a - r| <= 1e-5 |r| + 1e-5 max|r|); logits summed over C > 64 channels follow
test_gpu_fullsize.py's 720-channel rule (2e-5, and no worse than twice an fp32 comparator's distance from the fp64
value: the oracle in fp32 at full size, plain_conv elsewhere); bf16 dfeats (the fp32 value rounded once to nearest
even) is held to half a bf16 ulp on top of the 1e-5 bound."""
import pytest
import torch
import torch.nn.functional as F

from oracle import hier_oracle as O

DEV = "cuda"
BF = torch.bfloat16
CL = torch.channels_last
gpu = pytest.mark.gpu
SIGMOID, GROUPED, ZEROS = 0, 1, 2  # RHSEG_ACT_*
ACT_IDS = {SIGMOID: "sigmoid", GROUPED: "grouped", ZEROS: "zeros"}
DTYPES = [torch.float32, BF]
DT_IDS = ["fp32", "bf16"]
NAN = float("nan")


# ------------------------------------------------------------------------------------------------------------------
# part 0: the fp64 reference
# ------------------------------------------------------------------------------------------------------------------
def ref_fold(head_w, head_b, film_w, film_b, prev_probs):
    """FiLM folded into the head conv: cond = mean P_prev, [gamma|beta] = film_w cond + film_b,
    eff_w[b,k,c] = head_w[k,c] gamma[b,c], eff_b[b,k] = head_b[k] + sum_c head_w[k,c] beta[b,c]."""
    C = head_w.shape[1]
    hw = head_w.reshape(head_w.shape[0], C)
    gb = prev_probs.mean(dim=(2, 3)) @ film_w.T + film_b
    return hw[None] * gb[:, None, :C], head_b[None] + gb[:, C:] @ hw.T


def einsum_conv(ew, f, eb):
    return torch.einsum("bkc,bchw->bkhw", ew, f) + eb[:, :, None, None]


def plain_conv(ew, f, eb):
    """the same 1x1 conv summed one channel at a time in ascending order: in fp32 this is the plain fp32 comparator of
    the 720-channel rule (a BLAS kernel sums in blocks and carries less rounding error than any per-pixel chain)"""
    z = eb[:, :, None, None].expand(-1, -1, *f.shape[2:])
    for c in range(f.shape[1]):
        z = z + ew[:, :, c, None, None] * f[:, None, c]
    return z


def ref_level(f, eff_w, eff_b, act, prev_probs=None, parent=None, out_size=None, conv=einsum_conv):
    """One level forward: z = eff_w . f + eff_b ([K,C] / [K] weights are shared by all samples), bilinear
    align_corners upsample to out_size, then sigmoid / P_parent * softmax(z_g + log(P_parent + GATE_EPS)) over each run
    of channels with the same parent / zeros.  Returns logits, probs and psum = sum over pixels of probs."""
    ew = eff_w if eff_w.dim() == 3 else eff_w.expand(f.shape[0], -1, -1)
    eb = eff_b if eff_b.dim() == 2 else eff_b.expand(f.shape[0], -1)
    z = conv(ew, f, eb)
    if out_size is not None and tuple(out_size) != tuple(f.shape[2:]):
        z = F.interpolate(z, size=tuple(out_size), mode="bilinear", align_corners=True)
    if act == SIGMOID:
        p = torch.sigmoid(z)
    elif act == ZEROS:
        p = torch.zeros_like(z)
    else:
        pieces, k0 = [], 0
        while k0 < len(parent):
            k1 = k0
            while k1 < len(parent) and parent[k1] == parent[k0]:
                k1 += 1
            pp = prev_probs[:, parent[k0]:parent[k0] + 1]
            pieces.append(pp * torch.softmax(z[:, k0:k1] + torch.log(pp + O.GATE_EPS), dim=1))
            k0 = k1
        p = torch.cat(pieces, dim=1)
    return z, p, p.sum(dim=(2, 3))


def ref_conv_bwd(f, dz, eff_w):
    """1x1-conv backward: dfeats = sum_k eff_w dz, S = sum_n dz f, s = sum_n dz."""
    ew = eff_w if eff_w.dim() == 3 else eff_w.expand(f.shape[0], -1, -1)
    return torch.einsum("bkc,bkhw->bchw", ew, dz), torch.einsum("bkhw,bchw->bkc", dz, f), dz.sum(dim=(2, 3))


def ref_head(tree_dict, feats, hw, hb, fw, fb, out_size=None, conv=einsum_conv):
    """The whole head from the two functions above (FiLM fold, then one level at a time)."""
    levels, parent_of, _, groups = O.hierarchy_tables(tree_dict)
    probs, logits = [], []
    for L in range(len(levels)):
        if L == 0:
            ew, eb = hw[0].reshape(hw[0].shape[0], -1), hb[0]
            act, parent = SIGMOID, None
        else:
            ew, eb = ref_fold(hw[L], hb[L], fw[L - 1], fb[L - 1], probs[L - 1])
            parent = [levels[L - 1].index(parent_of[c]) for _, kids in groups[L - 1] for c in kids]
            act = GROUPED if groups[L - 1] else ZEROS
        z, p, _ = ref_level(feats[L], ew, eb, act, probs[L - 1] if L else None, parent, out_size, conv)
        logits.append(z)
        probs.append(p)
    return probs, logits


TL = {"background": {}, "upper": {}, "lower": {}, "tooth": {"pulp": {}, "dentin": {}, "enamel": {}, "composite": {}}}
EXT = {"background": {}, "tooth+alveolar": {"alveolar": {"upper": {}, "lower": {}},
                                            "tooth": {"composite": {}, "healthy": {"pulp": {}, "dentin": {}, "enamel": {}}}}}


@pytest.mark.parametrize("out_size", [None, (13, 17)], ids=["fullres", "upsampled"])
@pytest.mark.parametrize("tree", [TL, EXT], ids=["tl", "ext"])
def test_fp64_reference_reproduces_the_oracle_head(tree, out_size):
    levels, _, _, groups = O.hierarchy_tables(tree)
    chans = [len(levels[0])] + [sum(len(k) for _, k in g) for g in groups]
    g = torch.Generator().manual_seed(11)
    B, C, h, w = 2, 6, 5, 7
    d = torch.float64
    feats = [torch.randn(B, C, h, w, generator=g, dtype=d) for _ in chans]
    hw = [torch.randn(k, C, 1, 1, generator=g, dtype=d) * 0.4 for k in chans]
    hb = [torch.randn(k, generator=g, dtype=d) * 0.2 for k in chans]
    fw = [torch.randn(2 * C, kp, generator=g, dtype=d) * 0.6 for kp in chans[:-1]]
    fb = [torch.randn(2 * C, generator=g, dtype=d) * 0.3 + 1.0 for _ in chans[:-1]]
    p_o, z_o = O.head_forward(feats, hw, hb, fw, fb, levels, groups, out_size)
    p_r, z_r = ref_head(tree, feats, hw, hb, fw, fb, out_size)
    for L in range(len(chans)):
        torch.testing.assert_close(z_r[L], z_o[L], rtol=1e-12, atol=1e-12)
        torch.testing.assert_close(p_r[L], p_o[L], rtol=1e-12, atol=1e-12)


def test_fp64_conv_backward_reference_is_the_adjoint():
    g = torch.Generator().manual_seed(12)
    B, C, K, h, w = 2, 5, 3, 4, 6
    f = torch.randn(B, C, h, w, generator=g, dtype=torch.float64, requires_grad=True)
    ew = torch.randn(B, K, C, generator=g, dtype=torch.float64, requires_grad=True)
    eb = torch.randn(B, K, generator=g, dtype=torch.float64, requires_grad=True)
    dz = torch.randn(B, K, h, w, generator=g, dtype=torch.float64)
    z, _, _ = ref_level(f, ew, eb, ZEROS)
    z.backward(dz)
    dfeats, S, s = ref_conv_bwd(f.detach(), dz, ew.detach())
    torch.testing.assert_close(dfeats, f.grad, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(S, ew.grad, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(s, eb.grad, rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------------------------------------------------------
# shared pieces of the device tests
# ------------------------------------------------------------------------------------------------------------------
def is_cl(t):
    return t.is_contiguous(memory_format=CL) and not t.is_contiguous()


def bf16_values(*shape, gen, scale=1.0):
    """fp32 values that bf16 holds exactly (device tensor)"""
    return (torch.randn(*shape, generator=gen, device=DEV) * scale).to(BF).float()


def feats_as(base, dtype, layout):
    """base (fp32, bf16-representable, NCHW) as the kernels read it, and the call's feature flags.  Asserts the
    precondition of the flag: NHWC = channels-last in memory, 16-byte pixels and base."""
    from rhseg_b200 import native
    f = base.detach().to(dtype).clone(memory_format=CL if layout == "nhwc" else torch.contiguous_format)
    flag = native.FEATS_BF16 if dtype == BF else 0
    if layout == "nhwc":
        assert (f.shape[1] == 1 or f.shape[2] * f.shape[3] == 1 or is_cl(f)) and f.stride(1) == 1
        assert (f.shape[1] * f.element_size()) % 16 == 0 and f.data_ptr() % 16 == 0
        flag |= native.FEATS_NHWC
    else:
        assert f.is_contiguous()
    return f, flag


def close(a, ref, rtol=1e-5, what=""):
    """helpers.close's bound, |a - ref| <= rtol |ref| + rtol max|ref|, evaluated on the device (the tensors of the
    flush test hold 10^8 elements)"""
    a, ref = a.detach().double(), ref.detach().to(a.device).double()
    assert a.shape == ref.shape, (what, a.shape, ref.shape)
    if ref.numel() == 0:
        return
    err = (a - ref).abs()
    bad = ~(err <= rtol * ref.abs() + rtol * ref.abs().max() + 1e-12)  # a NaN is out of tolerance
    assert not bool(bad.any()), "%s: %d/%d out of tolerance, max err %.3e (scale %.3e)" % (
        what, int(bad.sum()), ref.numel(), err.max().item(), ref.abs().max().item())


def close_wide(got, ref64, ref32, what):
    """test_gpu_fullsize.py's rule for fp32 dot products over many channels: 2e-5, and no worse than twice the fp32
    comparator's own distance from the fp64 value"""
    close(got, ref64, rtol=2e-5, what=what)
    e = (got.detach().double() - ref64.double()).abs().max().item()
    e32 = (ref32.double() - ref64.double()).abs().max().item()
    assert e <= 2.0 * e32, (what, e, e32)


def close_bf16(got, ref, what):
    """a bf16 store of an fp32 value that is within 1e-5 of ref: half a bf16 ulp more"""
    a, r = got.detach().double(), ref.detach().to(got.device).double()
    bad = ~((a - r).abs() <= 2.0 ** -8 * r.abs() + 1e-5 * r.abs() + 1e-5 * r.abs().max() + 1e-12)
    assert not bool(bad.any()), "%s: %d/%d out of tolerance, max err %.3e" % (what, int(bad.sum()), r.numel(),
                                                                             (a - r).abs().max().item())


class no_tf32:
    """fp32 comparators without TF32 (cuDNN convolutions default to it)"""

    def __enter__(self):
        self.saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False

    def __exit__(self, *a):
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = self.saved
        return False


def parents(K, K_prev):
    """parent channel of each of K channels: contiguous runs over K_prev parents (groups of unequal size)"""
    return [k * K_prev // K for k in range(K)]


def table_of(act, K, K_prev):
    from rhseg_b200 import native
    tab = native.compile_level_table(parents(K, K_prev) if act != SIGMOID else [-1] * K, K_prev if act != SIGMOID else 0)
    return torch.tensor(tab, dtype=torch.int32, device=DEV)


def level_fwd(f, flag, eff_w, eff_b, act, K_prev=0, prev=None, out_size=None, z_lo=None, extra=0):
    """rhseg_head_level_fwd on fresh NaN-filled outputs; eff_w [K,C] (flag 4: shared by all samples) or [B,K,C]"""
    from rhseg_b200.native import call, ptr, stream_of
    B, C, Hf, Wf = f.shape
    K = eff_w.shape[-2]
    H, W = out_size if out_size is not None else (Hf, Wf)
    logits = torch.full((B, K, H, W), NAN, device=DEV)
    probs = torch.full((B, K, H, W), NAN, device=DEV)
    psum = torch.full((B, K), NAN, dtype=torch.float64, device=DEV)
    shared = 4 if eff_w.dim() == 2 else 0
    call("rhseg_head_level_fwd", ptr(f), ptr(eff_w), ptr(eff_b), ptr(prev), ptr(table_of(act, K, K_prev)), B, C, Hf, Wf,
         H, W, K, K_prev, act, ptr(z_lo), ptr(logits), ptr(probs), ptr(psum), 1 | shared | flag | extra, stream_of(f))
    return logits, probs, psum


def conv_bwd(f, flag, dz, eff_w, want_dfeats=True):
    """rhseg_head_conv_bwd; dfeats NaN-filled in the layout of f, or NULL"""
    from rhseg_b200.native import call, ptr, stream_of
    B, C = f.shape[:2]
    K = dz.shape[1]
    df = torch.full_like(f, NAN) if want_dfeats else None
    S = torch.full((B, K, C), NAN, dtype=torch.float64, device=DEV)
    s = torch.full((B, K), NAN, dtype=torch.float64, device=DEV)
    shared = 2 if eff_w.dim() == 2 else 0
    call("rhseg_head_conv_bwd", ptr(f), ptr(dz), ptr(eff_w), B, C, K, f.shape[2] * f.shape[3], ptr(df), ptr(S), ptr(s),
         1 | shared | flag, stream_of(f))
    return df, S, s


def check_fwd(what, got, ref, wide=False, ref32=None):
    z, p, ps = got
    zr, pr, psr = ref
    if wide:
        close_wide(z, zr, ref32, what + " logits")
        close(p, pr, rtol=2e-5, what=what + " probs")
        close(ps, psr, rtol=2e-5, what=what + " psum")
    else:
        close(z, zr, what=what + " logits")
        close(p, pr, what=what + " probs")
        close(ps, psr, what=what + " psum")


def check_bwd(what, got, ref, dtype, layout):
    df, S, s = got
    dr, Sr, sr = ref
    if df is not None:
        if layout == "nhwc":
            assert is_cl(df) or df.shape[1] == 1 or df.shape[2] * df.shape[3] == 1, what + " dfeats layout"
        (close_bf16 if dtype == BF else close)(df, dr, what=what + " dfeats")
    close(S, Sr, what=what + " S")
    close(s, sr, what=what + " s")


def kernel_names(fn):
    """CUDA kernel names launched by fn() (torch.profiler)"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def instances(names, kernel, dtype):
    """distinct instances of a templated kernel with the given feature element type among the launched names"""
    ft = "float" if dtype == torch.float32 else "unsigned short"
    return {n for n in names if "%s<%s," % (kernel, ft) in n}


def run_checks(checks):
    """runs every check, collects the failures: one report for a whole sweep"""
    bad = []
    for what, fn in checks:
        try:
            fn()
        except AssertionError as e:
            bad.append("%s: %s" % (what, str(e).splitlines()[0]))
    return bad


# ------------------------------------------------------------------------------------------------------------------
# part 1: every kernel instance through the C-ABI
# ------------------------------------------------------------------------------------------------------------------
SWEEP_B, SWEEP_C = 2, 40      # 160-byte (fp32) / 80-byte (bf16) pixels: 5 full stages of 8 channels
PLANES = {"v4": (40, 44),     # N = 1760, a multiple of 8: 16-byte rows in both dtypes (V4 tiles, NHWC: XCHG epilogue)
          "s1": (37, 41)}     # N = 1517, odd: scalar rows (S1 tiles); several tiles per sample, the last one partial
LOWRES_OUT = {"v4": (61, 70), "s1": (55, 62)}
K_PREV = 3


def _sweep(dtype, layout):
    """all level-forward and conv-backward calls of the sweep, each with its fp64 reference; returns the checks"""
    gen = torch.Generator(device=DEV).manual_seed(2024 + (dtype == BF) + 2 * (layout == "nhwc"))
    B, C = SWEEP_B, SWEEP_C
    checks = []
    for plane, (h, w) in PLANES.items():
        N = h * w
        assert (N % 8 == 0) if plane == "v4" else (N % 2 == 1), "tile-shape precondition"
        base = bf16_values(B, C, h, w, gen=gen)
        f, flag = feats_as(base, dtype, layout)
        f64 = base.double()
        for K in range(1, 9):
            # forward at feature resolution, every activation; weights per sample for odd K, shared (flag 4) for even K
            for act in (SIGMOID, GROUPED, ZEROS):
                shared = K % 2 == 0
                ew = bf16_values(*(((K, C) if shared else (B, K, C))), gen=gen, scale=0.3)
                eb = bf16_values(*(((K,) if shared else (B, K))), gen=gen, scale=0.5)
                kp = 0 if act == SIGMOID else K_PREV
                prev = torch.rand(B, K_PREV, h, w, generator=gen, device=DEV) * 0.9 + 0.05 if act == GROUPED else None
                got = level_fwd(f, flag, ew, eb, act, kp, prev)
                ref = ref_level(f64, ew.double(), eb.double(), act, prev.double() if prev is not None else None,
                                parents(K, K_PREV))
                checks.append(("fwd %s K=%d %s" % (plane, K, ACT_IDS[act]), lambda g=got, r=ref: check_fwd("", g, r)))
            # low-resolution conv (MODE_CONV_ONLY) + the hi-res pass, per-sample weights, z_lo zeroed by the call
            act = (SIGMOID, GROUPED, ZEROS)[K % 3]
            out = LOWRES_OUT[plane]
            ew = bf16_values(B, K, C, gen=gen, scale=0.3)
            eb = bf16_values(B, K, gen=gen, scale=0.5)
            kp = 0 if act == SIGMOID else K_PREV
            prev = torch.rand(B, K_PREV, *out, generator=gen, device=DEV) * 0.9 + 0.05 if act == GROUPED else None
            z_lo = torch.full((B, K, h, w), NAN, device=DEV)
            got = level_fwd(f, flag, ew, eb, act, kp, prev, out_size=out, z_lo=z_lo)
            ref = ref_level(f64, ew.double(), eb.double(), act, prev.double() if prev is not None else None,
                            parents(K, K_PREV), out)
            zlo_ref = ref_level(f64, ew.double(), eb.double(), ZEROS)[0]
            checks.append(("lowres %s K=%d z_lo" % (plane, K), lambda a=z_lo, r=zlo_ref: close(a, r)))
            checks.append(("lowres %s K=%d %s" % (plane, K, ACT_IDS[act]), lambda g=got, r=ref: check_fwd("", g, r)))
            # conv backward: per-sample and shared (flag 2) weights, and without dfeats
            dz = torch.randn(B, K, h, w, generator=gen, device=DEV)
            for shared in (False, True):
                ew = bf16_values(*(((K, C) if shared else (B, K, C))), gen=gen, scale=0.3)
                got = conv_bwd(f, flag, dz, ew)
                ref = ref_conv_bwd(f64, dz.double(), ew.double())
                checks.append(("bwd %s K=%d %s" % (plane, K, "shared" if shared else "per-sample"),
                               lambda g=got, r=ref: check_bwd("", g, r, dtype, layout)))
            if plane == "v4":
                got = conv_bwd(f, flag, dz, ew, want_dfeats=False)
                checks.append(("bwd %s K=%d dfeats=NULL" % (plane, K),
                               lambda g=got, r=ref: check_bwd("", g, r, dtype, layout)))
    return checks


# instances the sweep launches: NHWC forward = K x 3 activations x {XCHG, S1} + K low-res (S1 only), backward = K;
# NCHW forward = K x 3 activations x {V4, S1} + K low-res x {V4, S1}, backward = K x {V4, S1}
EXPECTED = {"nhwc": {"head_fwd_nhwc_kernel": 8 * 3 * 2 + 8, "conv_bwd_nhwc_kernel": 8},
            "nchw": {"head_fwd_kernel": 8 * 3 * 2 + 8 * 2, "conv_bwd_kernel": 8 * 2}}


@gpu
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_every_kernel_instance_against_fp64(dtype, layout):
    """All four dtype x layout combinations together launch the 128 NHWC instances (56 forward + 8 backward per
    dtype) and 160 NCHW ones."""
    out = {}
    names = kernel_names(lambda: out.setdefault("checks", _sweep(dtype, layout)))
    bad = run_checks(out["checks"])
    assert not bad, "%d of %d checks failed:\n%s" % (len(bad), len(out["checks"]), "\n".join(bad))
    for kernel, want in EXPECTED[layout].items():
        got = instances(names, kernel, dtype)
        assert len(got) == want, (kernel, len(got), want, sorted(got))
    other = "nchw" if layout == "nhwc" else "nhwc"
    for kernel in EXPECTED[other]:  # the flag reached the path it names, and only that one
        assert not instances(names, kernel, dtype), kernel


# ------------------------------------------------------------------------------------------------------------------
# part 2: persistent-grid paths and the edges of the NHWC contract
# ------------------------------------------------------------------------------------------------------------------
# Grids (launchers in head_fwd_kernel.cuh, head_fwd_nhwc.cuh, head_bwd_nhwc.cu): grid = min(SMs x CTAs per SM, work),
# the work split evenly over the grid.  CTAs per SM are at most min(threads per SM / block threads, shared memory per SM
# / the CTA's shared memory); registers can only lower it.  The preconditions below hold for EVERY CTA count per SM up to
# that bound, so they hold for whatever the device picks.
def _pad_k(K):
    return 1 if K <= 1 else 2 if K <= 2 else 4 if K <= 4 else 8


def fwd_geometry(dtype, layout, plane, C, K, N):
    """(tile pixels T, channels per stage, CTA threads, CTA shared memory) of the level-forward conv launch.
    plane: "v4" (16-byte rows), "s1" (scalar rows) or "lowres" (MODE_CONV_ONLY on scalar rows)."""
    esz = 4 if dtype == torch.float32 else 2
    J = 2 if esz == 4 else 4   # scalar-row tiles: T = 128 J (both layouts)
    KP = _pad_k(K)
    if layout == "nhwc":
        if plane == "v4":    # FwdNhwcCfgV4 = PipeCfg<8, 8, 3>: 8 consumer warps x 4 px, XCHG epilogue buffer
            T, NS, ncw, threads, xchg = 1024, 3, 8, 288, 1024
        else:                # FwdNhwcCfgS1 = PipeCfg<4, 8, 8, 2>
            T, NS, ncw, threads, xchg = 128 * J, 8, 4, 192, 0
        return T, 8, threads, 1024 + 128 + NS * T * 8 * esz + (C * KP + ncw * K + xchg) * 4
    G = 16 // esz
    if plane == "v4":        # FwdCfgV4 = PipeCfg<8, 8, 3>
        T, CH, NS, ncw, threads = 1024, 8, 3, 8, 288
    else:                    # FwdCfgS1 = PipeCfg<4, 16, 4, 2>
        T, CH, NS, ncw, threads = 128 * J, 16, 4, 4, 192
    return T, CH, threads, 128 + NS * CH * (T + G) * esz + (C * KP + ncw * K) * 4


def bwd_nhwc_geometry(dtype, C, N, B):
    """(pixels per tile TP, units, CTA threads, CTA shared memory) of conv_bwd_nhwc_kernel"""
    esz = 4 if dtype == torch.float32 else 2
    VC = 16 // esz
    NG = C // VC
    PL = 256 // NG
    ncons = (PL * NG + 31) // 32 * 32
    TP = max(PL, (24576 // (C * esz)) // PL * PL)
    return TP, B * -(-N // TP), ncons + 32, 128 + 4 * TP * C * esz + ncons * (VC + 1) * 4


def max_ctas_per_sm(threads, smem):
    p = torch.cuda.get_device_properties(0)
    return p.multi_processor_count, min(p.max_threads_per_multi_processor // threads, p.shared_memory_per_multiprocessor // smem)


def _grids(threads, smem, work):
    sms, bound = max_ctas_per_sm(threads, smem)
    assert bound >= 1
    return [min(sms * k, work) for k in range(1, bound + 1)]


# --- forward: a CTA's tiles span a sample boundary (psum flush, weight / bias reload) ----------------------------
SAMPLE_CHANGE = {"v4": (7, 64, 512, 521),   # B, C, h, w: N = 266 752 (multiple of 8), 261 tiles of 1024 px per sample
                 "s1": (5, 64, 511, 263)}   # N = 134 393 (odd): 525 (fp32) / 263 (bf16) tiles per sample


@gpu
@pytest.mark.parametrize("plane", ["v4", "s1"])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_forward_sample_change_inside_a_cta(dtype, layout, plane):
    B, C, h, w = SAMPLE_CHANGE[plane]
    N, K = h * w, 4
    T, _, threads, smem = fwd_geometry(dtype, layout, plane, C, K, N)
    n_tiles = -(-N // T)
    tiles = B * n_tiles
    grids = _grids(threads, smem, tiles)
    assert tiles >= 2 * max(grids), (tiles, grids)  # every CTA owns two tiles or more
    for grid in grids:  # and some CTA's tile range crosses from one sample into the next
        spans = [(tiles * i // grid, tiles * (i + 1) // grid) for i in range(grid)]
        assert any(t0 // n_tiles != (t1 - 1) // n_tiles for t0, t1 in spans), grid
    gen = torch.Generator(device=DEV).manual_seed(77)
    base = bf16_values(B, C, h, w, gen=gen)
    f, flag = feats_as(base, dtype, layout)
    # per-sample weights and biases far apart: a stale reload of the previous sample's shows at once
    ew = bf16_values(B, K, C, gen=gen, scale=0.2) + torch.arange(B, device=DEV).view(B, 1, 1) * 0.05
    eb = bf16_values(B, K, gen=gen) + torch.arange(B, device=DEV).view(B, 1) * 0.5
    prev = torch.rand(B, K_PREV, h, w, generator=gen, device=DEV) * 0.9 + 0.05
    got = level_fwd(f, flag, ew, eb, GROUPED, K_PREV, prev)
    del f
    ref = ref_level(base.double(), ew.double(), eb.double(), GROUPED, prev.double(), parents(K, K_PREV))
    check_fwd("%s/%s/%s" % (dtype, layout, plane), got, ref)


# --- low-res conv: tiles split between two CTAs (atomics into z_lo), with and without the caller's zero fill ----------
@gpu
@pytest.mark.parametrize("zeroed", [False, True], ids=["zlo_by_the_call", "zlo_zeroed_by_caller"])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_lowres_conv_split_tiles(dtype, layout, zeroed):
    B, C, h, w, K, out = 8, 720, 155, 155, 4, (620, 620)   # HRNet-W48's low-res plane, odd: scalar rows
    N = h * w
    T, CH, threads, smem = fwd_geometry(dtype, layout, "lowres", C, K, N)
    tiles, n_stages = B * -(-N // T), -(-C // CH)
    units = tiles * n_stages
    for grid in _grids(threads, smem, tiles):  # some CTA boundary falls inside a tile
        assert any(units * i // grid % n_stages for i in range(1, grid)), grid
    gen = torch.Generator(device=DEV).manual_seed(78)
    base = bf16_values(B, C, h, w, gen=gen)
    f, flag = feats_as(base, dtype, layout)
    ew = bf16_values(B, K, C, gen=gen, scale=C ** -0.5)
    eb = bf16_values(B, K, gen=gen, scale=0.5)
    prev = torch.rand(B, K_PREV, *out, generator=gen, device=DEV) * 0.9 + 0.05
    # bit 1 of the flags: z_lo is zero on entry; without it the call must zero it (a NaN would survive otherwise)
    z_lo = torch.zeros(B, K, h, w, device=DEV) if zeroed else torch.full((B, K, h, w), NAN, device=DEV)
    got = level_fwd(f, flag, ew, eb, GROUPED, K_PREV, prev, out_size=out, z_lo=z_lo, extra=2 if zeroed else 0)
    f64 = base.double()
    zr = ref_level(f64, ew.double(), eb.double(), ZEROS)[0]
    z32 = ref_level(base, ew, eb, ZEROS, conv=plain_conv)[0]
    close_wide(z_lo, zr, z32, "z_lo")
    ref = ref_level(f64, ew.double(), eb.double(), GROUPED, prev.double(), parents(K, K_PREV), out)
    z32 = F.interpolate(z32, size=out, mode="bilinear", align_corners=True)  # fp32, as the oracle's fp32 path
    check_fwd("%s/%s" % (dtype, layout), got, ref, wide=True, ref32=z32)


# --- conv backward: more than FLUSH_UNITS = 64 units per CTA --------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_conv_backward_flushes_within_a_sample(dtype):
    B, C, h, w, K = 2, 64, 1024, 2048, 4
    N = h * w
    TP, units, threads, smem = bwd_nhwc_geometry(dtype, C, N, B)
    grids = _grids(threads, smem, units)
    assert units // max(grids) > 64, (units, grids)  # every CTA flushes at least once before its sample ends
    gen = torch.Generator(device=DEV).manual_seed(79)
    base = bf16_values(B, C, h, w, gen=gen)
    f, flag = feats_as(base, dtype, "nhwc")
    dz = torch.randn(B, K, h, w, generator=gen, device=DEV)
    ew = bf16_values(B, K, C, gen=gen, scale=0.3)
    got = conv_bwd(f, flag, dz, ew)
    del f
    check_bwd(str(dtype), got, ref_conv_bwd(base.double(), dz.double(), ew.double()), dtype, "nhwc")


# --- channel counts at the edges of the contract ----------------------------------------------------------------------
EDGE_C = [(torch.float32, 4),     # 16-byte pixel: narrower than the 8-channel box
          (torch.float32, 12),    # a partial last stage (4 channels) under the 32-byte swizzle
          (torch.float32, 1020), (torch.float32, 1024),   # up to the 4096-byte pixel: NG = 256, PL = 1, TP = 6
          (BF, 8), (BF, 2040), (BF, 2048)]
EDGE_PLANES = {"v4": (40, 44), "s1": (37, 41), "row": (1, 300), "col": (301, 1)}


@gpu
@pytest.mark.parametrize("plane", list(EDGE_PLANES))
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("dtype,C", EDGE_C, ids=["%s-C%d" % ("fp32" if d == torch.float32 else "bf16", c) for d, c in EDGE_C])
def test_channel_counts_at_the_edges(dtype, C, layout, plane):
    B = 2
    h, w = EDGE_PLANES[plane]
    gen = torch.Generator(device=DEV).manual_seed(C + h)
    base = bf16_values(B, C, h, w, gen=gen)
    f, flag = feats_as(base, dtype, layout)
    f64 = base.double()
    wide = C > 64
    sc = C ** -0.5
    checks = []
    # forward at feature resolution, K = 8, grouped, per-sample weights
    K = 8
    ew = bf16_values(B, K, C, gen=gen, scale=sc)
    eb = bf16_values(B, K, gen=gen, scale=0.5)
    prev = torch.rand(B, K_PREV, h, w, generator=gen, device=DEV) * 0.9 + 0.05
    got = level_fwd(f, flag, ew, eb, GROUPED, K_PREV, prev)
    ref = ref_level(f64, ew.double(), eb.double(), GROUPED, prev.double(), parents(K, K_PREV))
    z32 = ref_level(base, ew, eb, ZEROS, conv=plain_conv)[0] if wide else None
    checks.append(("fwd", lambda: check_fwd("fwd", got, ref, wide, z32)))
    # low-res conv, K = 5, per-sample weights
    if plane in ("v4", "s1"):
        K, out = 5, (2 * h + 1, 2 * w - 1)
        ew2 = bf16_values(B, K, C, gen=gen, scale=sc)
        eb2 = bf16_values(B, K, gen=gen, scale=0.5)
        z_lo = torch.full((B, K, h, w), NAN, device=DEV)
        got2 = level_fwd(f, flag, ew2, eb2, SIGMOID, 0, None, out_size=out, z_lo=z_lo)
        zr = ref_level(f64, ew2.double(), eb2.double(), ZEROS)[0]
        ref2 = ref_level(f64, ew2.double(), eb2.double(), SIGMOID, out_size=out)
        if wide:
            z32l = ref_level(base, ew2, eb2, ZEROS, conv=plain_conv)[0]
            z32u = F.interpolate(z32l, size=out, mode="bilinear", align_corners=True)
            checks.append(("lowres z_lo", lambda: close_wide(z_lo, zr, z32l, "z_lo")))
        else:
            checks.append(("lowres z_lo", lambda: close(z_lo, zr, what="z_lo")))
        checks.append(("lowres", lambda: check_fwd("lowres", got2, ref2, wide, z32u if wide else None)))
    # conv backward, K = 8 per-sample weights and K = 3 shared weights (dfeats sums over the padded fourth channel)
    for K, shared in ((8, False), (3, True)):
        dz = torch.randn(B, K, h, w, generator=gen, device=DEV)
        ew3 = bf16_values(*((K, C) if shared else (B, K, C)), gen=gen, scale=sc)
        got3 = conv_bwd(f, flag, dz, ew3)
        ref3 = ref_conv_bwd(f64, dz.double(), ew3.double())
        checks.append(("bwd K=%d" % K, lambda g=got3, r=ref3: check_bwd("bwd", g, r, dtype, layout)))
    bad = run_checks(checks)
    assert not bad, "\n".join(bad)


@gpu
@pytest.mark.parametrize("dtype,C", [(torch.float32, 1028), (BF, 2056)], ids=["fp32-C1028", "bf16-C2056"])
def test_wider_pixels_are_refused_alike_by_the_abi_and_the_head(dtype, C):
    """A 4112-byte pixel is past the NHWC conv backward's 4096 bytes: the C-ABI refuses it, head._nhwc_native too, and
    the drop-in head copies such features to NCHW and still matches the fp64 reference."""
    import rhseg_b200
    from rhseg_b200 import head, native
    from rhseg_b200.native import ptr, stream_of
    B, h, w, K = 2, 9, 11, 4
    gen = torch.Generator(device=DEV).manual_seed(C)
    base = bf16_values(B, C, h, w, gen=gen)
    f, flag = feats_as(base, dtype, "nhwc")
    assert C * f.element_size() == 4112 and not head._nhwc_native(f)
    dz = torch.randn(B, K, h, w, generator=gen, device=DEV)
    ew = bf16_values(B, K, C, gen=gen, scale=C ** -0.5)
    df = torch.empty_like(f)
    S = torch.zeros(B, K, C, dtype=torch.float64, device=DEV)
    s = torch.zeros(B, K, dtype=torch.float64, device=DEV)
    rc = native.lib().rhseg_head_conv_bwd(ptr(f), ptr(dz), ptr(ew), B, C, K, h * w, ptr(df), ptr(S), ptr(s), 1 | flag,
                                          stream_of(f))
    assert rc == -2, (rc, native.status_string(rc))  # RHSEG_ERR_UNSUPPORTED
    # the drop-in head on these channels-last features
    tree = rhseg_b200.ClassTree(TL)
    chans = tree.head_channels
    feats = [f.detach().clone(memory_format=torch.preserve_format).requires_grad_(True)]
    feats.append(feats_as(bf16_values(B, C, h, w, gen=gen), dtype, "nhwc")[0].requires_grad_(True))
    hw = [(bf16_values(k, C, 1, 1, gen=gen, scale=C ** -0.5)).requires_grad_(True) for k in chans]
    hb = [bf16_values(k, gen=gen, scale=0.2).requires_grad_(True) for k in chans]
    fw = [bf16_values(2 * C, chans[0], gen=gen, scale=0.5).requires_grad_(True)]
    fb = [(bf16_values(2 * C, gen=gen, scale=0.2) + 1.0).requires_grad_(True)]
    assert all(is_cl(x) for x in feats)
    probs, logits = rhseg_b200.hier_head_forward(tree, feats, hw, hb, fw, fb)
    leaves64 = [[x.detach().double().requires_grad_(True) for x in grp] for grp in (feats, hw, hb, fw, fb)]
    p64, z64 = ref_head(TL, *leaves64)
    with torch.no_grad():
        _, z32 = ref_head(TL, *[[x.detach().float() for x in grp] for grp in (feats, hw, hb, fw, fb)], conv=plain_conv)
    wz = [torch.randn(z.shape, generator=gen, device=DEV) for z in logits]
    wp = [torch.randn(p.shape, generator=gen, device=DEV) for p in probs]
    sum((z * a).sum() + (p * b).sum() for z, p, a, b in zip(logits, probs, wz, wp)).backward()
    sum((z * a.double()).sum() + (p * b.double()).sum() for z, p, a, b in zip(z64, p64, wz, wp)).backward()
    for L in range(2):
        close_wide(logits[L], z64[L].detach(), z32[L], "logits%d" % L)
        close(probs[L], p64[L].detach(), rtol=2e-5, what="probs%d" % L)
        (close_bf16 if dtype == BF else close)(feats[L].grad, leaves64[0][L].grad, what="dfeats%d" % L)
        close(hw[L].grad, leaves64[1][L].grad, what="dhead_w%d" % L)
        close(hb[L].grad, leaves64[2][L].grad, what="dhead_b%d" % L)
    close(fw[0].grad, leaves64[3][0].grad, what="dfilm_w")
    close(fb[0].grad, leaves64[4][0].grad, what="dfilm_b")


# ------------------------------------------------------------------------------------------------------------------
# part 3: the full-size workloads, fp32 / bf16 x NCHW / channels-last, against one fp64 oracle per workload
# ------------------------------------------------------------------------------------------------------------------
FULL = ["unet_tl_620_b4", "hrnet_w48_tl_620_b4", "hrnet_w48_ext_620_b4"]
_ORACLE = {}


def _full_oracle(name):
    """inputs (features rounded to bf16-representable values) and the fp64 oracle's loss, logits and gradients, on the
    GPU; the last workload's only (they are large)"""
    if name in _ORACLE:
        return _ORACLE[name]
    _ORACLE.clear()
    import bench
    wl = bench.WORKLOADS[name]
    B = wl["B"]
    # one sample without a tooth: its deeper-level Dice is NaN and is dropped (as in test_gpu_fullsize.py)
    data = bench.synth_inputs(wl, B, seed=3, device=DEV, notooth_sample=1)
    h = data["host"]
    h["feats"] = [f.to(BF).float() for f in h["feats"]]
    levels, parent_of, _, groups = O.hierarchy_tables(wl["tree"])
    out_size = None if wl["scale"] == 1 else (wl["H"], wl["W"])
    targets, s = [], 0
    for k in data["chans"]:
        targets.append(h["target"][:, s:s + k])
        s += k
    leaves = [[t.double().requires_grad_(True) for t in h[k]] for k in ("feats", "hw", "hb", "fw", "fb")]
    probs, logits = O.head_forward(*leaves, levels, groups, out_size)
    onehots, _ = O.predict_onehot_masked([z.detach().float() for z in logits], targets)
    loss, _ = O.total_loss(logits, targets, data["weights"], onehots, levels, parent_of)
    loss.backward()
    r = dict(wl=wl, data=data, targets=targets, out_size=out_size, loss=loss.item(),
             logits=[z.detach() for z in logits], probs=[p.detach() for p in probs],
             grads=[[t.grad for t in grp] for grp in leaves], logits32=None)
    del leaves, probs, logits, loss
    if wl["C"] > 64:  # the fp32 comparator of the 720-channel rule
        with no_tf32(), torch.no_grad():
            r["logits32"] = O.head_forward(*[h[k] for k in ("feats", "hw", "hb", "fw", "fb")], levels, groups, out_size)[1]
    _ORACLE[name] = r
    return r


@gpu
@pytest.mark.parametrize("name,dtype", [(n, d) for n in FULL for d in DTYPES],
                         ids=["%s-%s" % (n, i) for n in FULL for i in DT_IDS])
def test_full_size_feature_paths_against_the_fp64_oracle(name, dtype):
    import rhseg_b200
    from rhseg_b200 import head
    r = _full_oracle(name)
    wl, data, h = r["wl"], r["data"], r["data"]["host"]
    nL = len(data["chans"])
    wide = wl["C"] > 64
    step = rhseg_b200.FusedHierStep(wl["tree"], data["weights"])
    outs = {}
    for layout in ("nchw", "nhwc"):
        feats = [feats_as(f, dtype, layout)[0].requires_grad_(True) for f in h["feats"]]
        assert all(head._nhwc_native(f) == (layout == "nhwc") for f in feats)
        params = [[t.clone().requires_grad_(True) for t in h[k]] for k in ("hw", "hb", "fw", "fb")]
        out = step(feats, *params, h["target"], r["out_size"])
        out.loss.backward()
        what = "%s/%s/%s" % (name, DT_IDS[DTYPES.index(dtype)], layout)
        assert abs(out.loss.item() - r["loss"]) <= 1e-5 * abs(r["loss"]), (what, out.loss.item(), r["loss"])
        for L in range(nL):
            oh, et = O.predict_onehot_masked([out.logits[L]], [r["targets"][L]])
            want = O.level_confusion(oh[0], et[0], data["chans"][L], L != 0)
            assert torch.equal(out.confusion[L], want.to(out.confusion[L].device)), "%s confusion%d" % (what, L)
            if wide:
                close_wide(out.logits[L], r["logits"][L], r["logits32"][L], "%s logits%d" % (what, L))
            else:
                close(out.logits[L], r["logits"][L], what="%s logits%d" % (what, L))
            close(out.probs[L], r["probs"][L], rtol=2e-5 if wide else 1e-5, what="%s probs%d" % (what, L))
            g = feats[L].grad
            assert g.dtype == dtype and is_cl(g) == (layout == "nhwc"), what
            (close_bf16 if dtype == BF else close)(g, r["grads"][0][L], what="%s dfeats%d" % (what, L))
        for grp, rg, nm in zip(params, r["grads"][1:], ("dhead_w", "dhead_b", "dfilm_w", "dfilm_b")):
            for i, (p, pr) in enumerate(zip(grp, rg)):
                close(p.grad, pr, what="%s %s%d" % (what, nm, i))
        outs[layout] = out
        del feats, params
    # DESIGN.md 3.8: at feature resolution the fp32 channels-last logits and probabilities are the NCHW ones bit for bit
    # (both kernels get the same resident wave and split tiles alike); elsewhere they agree within the tolerance above
    if wl["scale"] == 1 and dtype == torch.float32:
        for L in range(nL):
            assert torch.equal(outs["nhwc"].logits[L], outs["nchw"].logits[L]), "logits%d" % L
            assert torch.equal(outs["nhwc"].probs[L], outs["nchw"].probs[L]), "probs%d" % L
