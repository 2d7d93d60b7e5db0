"""Restrictive-hierarchy head: all levels in ONE autograd node over the C-ABI kernels.

Forward per level (reference: Models/models.py:263-306 UNet, :757-802 HRNet):
    cond   = mean_{hw} P_{L-1}                     (psum of the previous level's kernel)
    z_L    = (W_L diag(gamma_b)) f_L + (W_L beta_b + bias_L)      FiLM folded into the 1x1 conv
    [z_L   = bilinear_up(z_L)]                      HRNet only
    P_0    = sigmoid(z_0);  P_L = P_parent * softmax_group(z_L)
Backward runs last level -> first (closed forms in DESIGN.md): the gradient reaching
P_{L-1} is a per-(sample, channel) constant from the FiLM pool plus, for trees deeper than two
levels, a per-pixel term from the composition.
"""
import os
from typing import List, Optional, Sequence, Tuple

import torch

from . import native
from .native import call, ptr, stream_of
from .tree_tables import ClassTree


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        raise native.NativeError("rhseg_b200 head expects float32 tensors, got %s" % t.dtype)
    return t if t.is_contiguous() else t.contiguous()


def _nhwc_native(f: torch.Tensor) -> bool:
    """Features the kernels read channels-last as they are (RHSEG_FEATS_NHWC): channels-last-contiguous but not
    contiguous (so C = 1 and 1x1 planes, which are both, keep the NCHW path), a pixel's channels a multiple of 16 bytes
    and at most 4096, a 16-byte aligned base."""
    if f.dim() != 4 or f.is_contiguous() or not f.is_contiguous(memory_format=torch.channels_last):
        return False
    row = f.shape[1] * f.element_size()
    return row % 16 == 0 and row <= 4096 and f.data_ptr() % 16 == 0


def _feats_flag(f: torch.Tensor) -> int:
    """Feature flags of the kernel calls for a tensor _feats_c returned: dtype, and layout (it returned only contiguous
    tensors and the channels-last ones the kernels read natively)."""
    return (native.FEATS_BF16 if f.dtype == torch.bfloat16 else 0) | (0 if f.is_contiguous() else native.FEATS_NHWC)


def _feats_c(feats: Sequence[torch.Tensor]) -> Tuple[List[torch.Tensor], List[int]]:
    """Per-level features as the kernels read them, and each level's flags (_feats_flag).  dtype: float32, or bfloat16
    on every level (donors trained under torch.autocast; the kernels convert each value to fp32 exactly and store dfeats
    as bf16).  Layout, per level: channels-last features (donors converted with torch.channels_last) are read in place
    when _nhwc_native allows it, and their dfeats comes back channels-last; anything else is made contiguous."""
    dt = feats[0].dtype
    if dt not in (torch.float32, torch.bfloat16) or any(f.dtype != dt for f in feats):
        raise native.NativeError("rhseg_b200 head expects float32 or bfloat16 features (one dtype for every level), got %s"
                                 % ", ".join(sorted({str(f.dtype) for f in feats})))
    out = [f if f.is_contiguous() or _nhwc_native(f) else f.contiguous() for f in feats]
    return out, [_feats_flag(f) for f in out]


_SIDE_STREAMS = {}
# Upsampled heads, fused training step: which levels are evaluated INSIDE their hi-res forward kernel
# (rhseg_head_level_fwd_eval) instead of by rhseg_level_eval on a side stream, concurrent with the next level's forward.
#   "last": only the last level (nothing is left to overlap with)     "root": also level 0     "all": every level
# Measured (DESIGN.md 6): HRNet-W48 tl "root" = "all" 0.420 ms vs "last" 0.428 ms; extended tree "all" is slower than "last".
_FUSE_EVAL = os.environ.get("RHSEG_FUSE_EVAL", "root")


def _side_stream(dev):
    """One auxiliary stream per device for kernels that are independent of the level chain."""
    key = (dev.type, dev.index)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=dev)
    return _SIDE_STREAMS[key]


def forward_levels(tree: ClassTree, out_size, tensors, evaluate=None, zero_words: int = 0, with_backward: bool = False):
    """Runs the per-level forward kernels.  `tensors` = feats[n] + head_w[n] + head_b[n] + film_w[n-1] +
    film_b[n-1]; the features are fp32 or bf16, contiguous or channels-last (_feats_c), everything else fp32.
    Returns a dict with the inputs (as the kernels read them) and probs / logits / psums / eff_w /
    gamma_beta per level plus the shape tuple.
    `evaluate(L, dims)` (fused training step) returns the rhseg_level_eval arguments of level L:
    (targets_ptr, t_bs, t_cs, parent_ptr, prev_idx_ptr, out_words_ptr, idx_out_ptr); the evaluation then runs
    inside the hi-res forward kernel (upsampled heads) or right after the level's forward (feature-resolution heads).
    `zero_words` extra fp64 words are zeroed by the same fill as the pool sums / low-res logits and handed to
    `evaluate` as its third argument (the fused step's statistics workspace).  with_backward: the same fill also
    zeroes the accumulators of the backward pass (r["bwd"], see backward_buffers): ONE fill per training step."""
    n = tree.num_levels
    feats, fflags = _feats_c(tensors[0:n])
    head_w = [_f32c(t) for t in tensors[n:2 * n]]
    head_b = [_f32c(t) for t in tensors[2 * n:3 * n]]
    film_w = [_f32c(t) for t in tensors[3 * n:4 * n - 1]]
    film_b = [_f32c(t) for t in tensors[4 * n - 1:5 * n - 2]]
    native.require_cuda(*feats, *head_w, *head_b, *film_w, *film_b)
    dev = feats[0].device
    st = stream_of(feats[0])
    tables = tree.device_tables(dev)
    B, C, Hf, Wf = feats[0].shape
    H, W = (Hf, Wf) if out_size is None else (int(out_size[0]), int(out_size[1]))
    upsampled = (H, W) != (Hf, Wf)
    n_pix = H * W
    probs, logits, psums, eff_ws, gbs = [], [], [], [], []
    # ONE zero fill per forward: every level's fp64 pool sums | the caller's workspace | the low-res logits of
    # all levels (fp32; tiles split between CTAs accumulate into them)
    n_psum = sum(tree.head_channels) * B
    n_zlo = B * sum(tree.head_channels) * Hf * Wf if upsampled else 0
    n_head = (n_psum + int(zero_words) + 1) // 2 * 2  # the fp32 tail starts 16-byte aligned, as a separate allocation would
    n_fwd = n_head + (n_zlo + 3) // 4 * 2
    n_bwd = backward_words(tree, B, C, (Hf, Wf) if upsampled else None) if with_backward else 0
    zero_all = torch.zeros((n_fwd + n_bwd,), dtype=torch.float64, device=dev)
    psum_all = zero_all[:n_psum]
    workspace = zero_all[n_psum:n_psum + int(zero_words)]
    zlo_all = zero_all[n_head:n_fwd].view(torch.float32) if upsampled else None
    bwd = backward_buffers(tree, B, C, dev, (Hf, Wf) if upsampled else None, zero_all[n_fwd:]) if with_backward else None
    psum_off = 0
    used_side = False
    zlo_off = 0
    for L in range(n):
        K = tree.head_channels[L]
        K_prev = tree.head_channels[L - 1] if L > 0 else 0
        f, fbf = feats[L], fflags[L]
        if tuple(f.shape) != (B, C, Hf, Wf):
            raise native.NativeError("per-level feature tensors must share one shape")
        if tuple(head_w[L].shape[:2]) != (K, C):
            raise native.NativeError("head weight of level %d has shape %s, expected [%d,%d,1,1]"
                                     % (L, tuple(head_w[L].shape), K, C))
        if L == 0:
            # no FiLM in front of level 0: the kernels read the head's own [K,C] weights (flag 4: shared by all samples)
            eff_w, eff_b, gb, shared = head_w[0], head_b[0], None, 4
        else:
            eff_w = torch.empty((B, K, C), dtype=torch.float32, device=dev)
            eff_b = torch.empty((B, K), dtype=torch.float32, device=dev)
            gb = torch.empty((B, 2 * C), dtype=torch.float32, device=dev)
            shared = 0
            call("rhseg_film_fold", ptr(head_w[L]), ptr(head_b[L]), ptr(film_w[L - 1]), ptr(film_b[L - 1]),
                 ptr(psums[L - 1]), float(n_pix), B, C, K, K_prev, ptr(gb), ptr(eff_w), ptr(eff_b), st)
        z = torch.empty((B, K, H, W), dtype=torch.float32, device=dev)
        p = torch.empty((B, K, H, W), dtype=torch.float32, device=dev)
        psum = psum_all[psum_off:psum_off + B * K].view(B, K)
        psum_off += B * K
        z_lo = None
        if upsampled:
            z_lo = zlo_all[zlo_off:zlo_off + B * K * Hf * Wf].view(B, K, Hf, Wf)
            zlo_off += B * K * Hf * Wf
        ev = evaluate(L, (B, C, Hf, Wf, H, W), workspace) if evaluate is not None else None
        hint = tree.group_hint(L)  # uniform group size: kernels with the group layout fixed at compile time
        # The evaluation of level L only needs its logits (and the previous level's index map): for all
        # but the last level it runs on a side stream, overlapping the (memory-bound) forward of the next
        # level; the last level's evaluation is fused into its hi-res forward kernel when there is one.
        overlap = ev is not None and L < n - 1 and not (upsampled and (_FUSE_EVAL == "all" or (_FUSE_EVAL == "root" and L == 0)))
        if ev is not None and upsampled and not overlap:
            t_ptr, t_bs, t_cs, pt_ptr, pidx_ptr, words_ptr, idx_ptr = ev
            if used_side:  # the previous level's index map is produced on the side stream
                torch.cuda.current_stream(dev).wait_stream(_side_stream(dev))
                used_side = False
            call("rhseg_head_level_fwd_eval", ptr(f), ptr(eff_w), ptr(eff_b),
                 ptr(probs[L - 1]) if L > 0 else None, ptr(tables[L]),
                 B, C, Hf, Wf, H, W, K, K_prev, tree.act_mode[L] | hint, ptr(z_lo), ptr(z), ptr(p), ptr(psum),
                 t_ptr, t_bs, t_cs, pt_ptr, t_bs, t_cs, pidx_ptr, words_ptr, idx_ptr, 1 | 2 | shared | fbf, st)
        else:
            call("rhseg_head_level_fwd", ptr(f), ptr(eff_w), ptr(eff_b),
                 ptr(probs[L - 1]) if L > 0 else None, ptr(tables[L]),
                 B, C, Hf, Wf, H, W, K, K_prev, tree.act_mode[L] | hint, ptr(z_lo), ptr(z), ptr(p), ptr(psum), (2 if upsampled else 0) | shared | fbf, st)
            if ev is not None:
                t_ptr, t_bs, t_cs, pt_ptr, pidx_ptr, words_ptr, idx_ptr = ev
                if overlap:
                    main = torch.cuda.current_stream(dev)
                    side = _side_stream(dev)
                    side.wait_stream(main)  # logits of this level (and everything before) are ready
                    call("rhseg_level_eval", ptr(z), t_ptr, t_bs, t_cs, pt_ptr, t_bs, t_cs, pidx_ptr, ptr(tables[L]),
                         B, K, n_pix, (1 if L > 0 else 0) | hint, words_ptr, idx_ptr, 1, side.cuda_stream)
                    used_side = True
                else:
                    if used_side:  # the previous level's index map is produced on the side stream
                        torch.cuda.current_stream(dev).wait_stream(_side_stream(dev))
                        used_side = False
                    call("rhseg_level_eval", ptr(z), t_ptr, t_bs, t_cs, pt_ptr, t_bs, t_cs, pidx_ptr, ptr(tables[L]),
                         B, K, n_pix, (1 if L > 0 else 0) | hint, words_ptr, idx_ptr, 1, st)
        probs.append(p); logits.append(z); psums.append(psum); eff_ws.append(eff_w); gbs.append(gb)
    if used_side:
        torch.cuda.current_stream(dev).wait_stream(_side_stream(dev))
    return dict(feats=feats, head_w=head_w, head_b=head_b, film_w=film_w, film_b=film_b, probs=probs, logits=logits,
                psums=psums, eff_ws=eff_ws, gbs=gbs, dims=(B, C, Hf, Wf, H, W), upsampled=upsampled, workspace=workspace, bwd=bwd)


def level_weight_backward(tree, L, dims, feats_L, dz_feat, eff_w_L, head_w_L, film_w_prev, gb_L, psum_prev, buf, want_dfeats, st):
    """conv backward + parameter gradients of one level given dz at feature resolution: ONE launch
    (rhseg_head_conv_bwd_params: the last CTA to finish forms the parameter gradients from the complete sums).
    `buf` = this level's entry of backward_buffers().  Returns (d_feats or None, d_head_w, d_head_b, d_film_w or None,
    d_film_b or None, g_prev or None)."""
    B, C, Hf, Wf, H, W = dims
    K = tree.head_channels[L]
    K_prev = tree.head_channels[L - 1] if L > 0 else 0
    dev = feats_L.device
    d_feats = torch.empty_like(feats_L) if want_dfeats else None
    d_hw = torch.empty_like(head_w_L)
    d_hb = torch.empty((K,), dtype=torch.float32, device=dev)
    d_fw = d_fb = g_prev = None
    if L > 0:
        d_fw = torch.empty_like(film_w_prev)
        d_fb = torch.empty((2 * C,), dtype=torch.float32, device=dev)
        g_prev = buf["gp"]
    fbf = _feats_flag(feats_L)  # d_feats: same dtype and layout as the features (empty_like keeps channels-last)
    call("rhseg_head_conv_bwd_params", ptr(feats_L), ptr(dz_feat), ptr(eff_w_L), B, C, K, Hf * Wf, ptr(d_feats),
         ptr(buf["S"]), ptr(buf["s"]), (2 if L == 0 else 0) | 4 | fbf, ptr(head_w_L), ptr(film_w_prev) if L > 0 else None, ptr(gb_L),
         ptr(psum_prev) if L > 0 else None, float(H * W), K_prev, ptr(d_hw), ptr(d_hb), ptr(d_fw), ptr(d_fb), ptr(g_prev),
         ptr(buf["ticket"]), st)
    return d_feats, d_hw, d_hb, d_fw, d_fb, g_prev


def _bwd_layout(tree, B, C, lowres_hw):
    """fp64 word offsets of the backward accumulators: per level S [B,K,C] | s [B,K] | g_prev [B,K_prev] | ticket, then
    (upsampled heads) one fp32 dz_lo [B,K,Hf,Wf] per level, each 16-byte aligned."""
    kprev = [0] + list(tree.head_channels[:-1])
    off, levels = 0, []
    for k, kp in zip(tree.head_channels, kprev):
        lv = dict(S=off, s=off + B * k * C, gp=off + B * k * (C + 1), ticket=off + B * k * (C + 1) + B * kp, k=k, kp=kp)
        off = lv["ticket"] + 1
        levels.append(lv)
    off += off & 1
    n_lo = 0 if lowres_hw is None else lowres_hw[0] * lowres_hw[1]
    for lv in levels:
        lv["dz"] = off
        off += (B * lv["k"] * n_lo + 3) // 4 * 2
    return levels, off


def backward_words(tree, B, C, lowres_hw=None):
    return _bwd_layout(tree, B, C, lowres_hw)[1]


def backward_buffers(tree, B, C, dev, lowres_hw=None, zeroed=None):
    """Zero-filled accumulators of the backward pass as per-level dicts of views: S, s, gp (pool-gradient accumulator,
    None at level 0), ticket (the conv kernel's last-CTA counter) and, with lowres_hw = (Hf, Wf), dz (the fp32 dz_lo the
    band adjoint adds into, RHSEG_DZ_PREZEROED).  `zeroed`: a zero fp64 tensor of backward_words() elements to carve the
    views from (the forward's single fill); otherwise one torch.zeros is made here."""
    levels, total = _bwd_layout(tree, B, C, lowres_hw)
    buf = zeroed if zeroed is not None else torch.zeros((total,), dtype=torch.float64, device=dev)
    out = []
    for lv in levels:
        k, kp = lv["k"], lv["kp"]
        d = dict(S=buf[lv["S"]:lv["S"] + B * k * C].view(B, k, C), s=buf[lv["s"]:lv["s"] + B * k].view(B, k),
                 gp=buf[lv["gp"]:lv["gp"] + B * kp].view(B, kp) if kp else None,
                 ticket=buf[lv["ticket"]:lv["ticket"] + 1].view(torch.int32), dz=None)
        if lowres_hw is not None:
            n = B * k * lowres_hw[0] * lowres_hw[1]
            d["dz"] = buf[lv["dz"]:lv["dz"] + (n + 3) // 4 * 2].view(torch.float32)[:n].view(B, k, lowres_hw[0], lowres_hw[1])
        out.append(d)
    return out


class _HierHeadFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, tree: ClassTree, out_size: Optional[Tuple[int, int]], *tensors):
        n = tree.num_levels
        grad = any(ctx.needs_input_grad)  # grad mode is off inside forward(): ask autograd
        r = forward_levels(tree, out_size, tensors, with_backward=grad)
        ctx.bwd = r["bwd"]
        feats, head_w, film_w = r["feats"], r["head_w"], r["film_w"]
        probs, logits, psums, eff_ws, gbs = r["probs"], r["logits"], r["psums"], r["eff_ws"], r["gbs"]
        ctx.tree, ctx.dims, ctx.upsampled = tree, r["dims"], r["upsampled"]
        ctx.save_for_backward(*feats, *head_w, *film_w, *logits, *probs, *psums, *eff_ws, *[g for g in gbs if g is not None])
        ctx.set_materialize_grads(False)
        outs = tuple(probs) + tuple(logits)
        return outs

    @staticmethod
    def backward(ctx, *grads):
        tree = ctx.tree
        n = tree.num_levels
        B, C, Hf, Wf, H, W = ctx.dims
        sv = ctx.saved_tensors
        feats, head_w, film_w = sv[0:n], sv[n:2 * n], sv[2 * n:3 * n - 1]
        o = 3 * n - 1
        logits, probs, psums, eff_ws = sv[o:o + n], sv[o + n:o + 2 * n], sv[o + 2 * n:o + 3 * n], sv[o + 3 * n:o + 4 * n]
        gbs = [None] + list(sv[o + 4 * n:o + 5 * n - 1])
        d_probs, d_logits = grads[0:n], grads[n:2 * n]
        dev = feats[0].device
        st = stream_of(feats[0])
        tables = tree.device_tables(dev)
        n_pix, n_feat = H * W, Hf * Wf

        d_feats: List[Optional[torch.Tensor]] = [None] * n
        d_hw: List[Optional[torch.Tensor]] = [None] * n
        d_hb: List[Optional[torch.Tensor]] = [None] * n
        d_fw: List[Optional[torch.Tensor]] = [None] * (n - 1)
        d_fb: List[Optional[torch.Tensor]] = [None] * (n - 1)

        # accumulators zeroed by the forward's fill; a second backward over the same graph gets fresh ones
        bufs, ctx.bwd = ctx.bwd, None
        if bufs is None:
            bufs = backward_buffers(tree, B, C, dev, (Hf, Wf) if ctx.upsampled else None)
        g_uniform = None   # [B,K_L] fp64: dLoss/d(sum_n P_L) * n_pix, from level L+1's FiLM
        dp_pix = None      # [B,K_L,H,W]: per-pixel dLoss/dP_L (composition of level L+1 and/or user grads)
        pix_mask = 0
        for L in range(n - 1, -1, -1):
            K = tree.head_channels[L]
            K_prev = tree.head_channels[L - 1] if L > 0 else 0
            mode = tree.act_mode[L]
            dz = d_logits[L]
            if dz is not None:
                dz = _f32c(dz)
            if d_probs[L] is not None:  # gradients a caller put directly on the probabilities
                if dp_pix is None:
                    dp_pix = _f32c(d_probs[L])
                else:
                    dp_pix = dp_pix + d_probs[L]
                pix_mask = (1 << K) - 1
            dp_prev, prev_mask = None, 0
            needs_act = mode != native.ACT_ZEROS and (g_uniform is not None or dp_pix is not None)
            if needs_act:
                dz_total = torch.empty((B, K, H, W), dtype=torch.float32, device=dev)
                if mode == native.ACT_GROUPED:
                    dp_prev = torch.zeros((B, K_prev, H, W), dtype=torch.float32, device=dev)
                    for pname, _ in tree.child_groups[L - 1]:
                        prev_mask |= 1 << tree.levels[L - 1].index(pname)
                call("rhseg_head_act_bwd", ptr(logits[L]), ptr(probs[L - 1]) if L > 0 else None, ptr(tables[L]),
                     ptr(dz), ptr(g_uniform), 1.0 / n_pix, ptr(dp_pix), pix_mask,
                     B, K, K_prev, H, W, mode, ptr(dz_total), ptr(dp_prev), st)
                dz = dz_total
            g_uniform, dp_pix, pix_mask = None, dp_prev, prev_mask
            if dz is None:
                continue  # nothing reaches this level's logits: no gradient for its features / parameters
            if ctx.upsampled:
                dz_lo = bufs[L]["dz"]  # zeroed together with the weight sums: the band adjoint adds into it
                call("rhseg_upsample_adjoint", ptr(dz), B, K, Hf, Wf, H, W, ptr(dz_lo), None, native.DZ_PREZEROED, st)
                dz = dz_lo
            d_feats[L], d_hw[L], d_hb[L], fw_g, fb_g, g_prev = level_weight_backward(
                tree, L, ctx.dims, feats[L], dz, eff_ws[L], head_w[L], film_w[L - 1] if L > 0 else None, gbs[L],
                psums[L - 1] if L > 0 else None, bufs[L], ctx.needs_input_grad[2 + L], st)
            if L > 0:
                d_fw[L - 1], d_fb[L - 1] = fw_g, fb_g
            g_uniform = g_prev
        return (None, None) + tuple(d_feats) + tuple(d_hw) + tuple(d_hb) + tuple(d_fw) + tuple(d_fb)


def hier_head_forward(tree: ClassTree, feats: Sequence[torch.Tensor],
                      head_w: Sequence[torch.Tensor], head_b: Sequence[torch.Tensor],
                      film_w: Sequence[torch.Tensor], film_b: Sequence[torch.Tensor],
                      out_size: Optional[Tuple[int, int]] = None):
    """(probs_per_level, logits_per_level), differentiable w.r.t. every input tensor.
    `feats[L]` is the donor backbone's feature map of its L-th pass [B,C,h,w]; `out_size`
    (H,W) != (h,w) selects the HRNet path (logits bilinearly upsampled, align_corners=True)."""
    n = tree.num_levels
    if not (len(feats) == len(head_w) == len(head_b) == n and len(film_w) == len(film_b) == n - 1):
        raise native.NativeError("hier_head_forward: expected %d levels of features/heads and %d FiLMs" % (n, n - 1))
    with native.device_guard(feats[0]):
        outs = _HierHeadFn.apply(tree, out_size, *feats, *head_w, *head_b, *film_w, *film_b)
    return list(outs[:n]), list(outs[n:])
