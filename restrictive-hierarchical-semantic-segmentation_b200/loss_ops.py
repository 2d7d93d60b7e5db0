"""Fused hierarchical-loss operators over the C-ABI kernels.

One autograd node per (logits, targets) pair yields BOTH the cross-entropy and the dice term
of a level from a single statistics pass, and back-propagates both through a single gradient
pass.  The reference's two loss modules (Metrics/losses.py:16-134) are called one after the
other on the same tensors (train.py:136-137); `level_loss` memoises on tensor identity so the
second module call reuses the node the first one created."""
import weakref
from typing import Optional, Sequence

import torch

from . import native
from .native import call, ptr, stream_of
from .tree_tables import tree_from_levels

_WEIGHTS = {}


def weight_tensor(class_weight: Sequence[float], device) -> torch.Tensor:
    """class_weight (python list, as train.py passes it) -> cached fp32 device tensor."""
    if class_weight is None:
        # the reference crashes here too (UnboundLocalError / TypeError, SURVEY.md F7)
        raise ValueError("class_weight=None is not supported by the reference losses; pass a list of K floats")
    key = (tuple(float(w) for w in class_weight), str(device))
    t = _WEIGHTS.get(key)
    if t is None:
        t = torch.tensor(key[0], dtype=torch.float32).to(device)
        _WEIGHTS[key] = t
    return t


def _plane_contiguous(t: torch.Tensor) -> torch.Tensor:
    """Targets arrive as channel slices target[:, s:e] (train.py:185-193): batch/channel strides
    are free, the H*W plane must be dense."""
    if t.dtype != torch.float32:
        t = t.float()
    if t.dim() == 4:
        ok = t.stride(3) == 1 and t.stride(2) == t.size(3)
    elif t.dim() == 3:
        ok = t.stride(2) == 1
    else:
        raise native.NativeError("targets must be [B,K,H,W] or [B,K,N]")
    return t if ok else t.contiguous()


class _LevelLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, outs, targets, weights, smooth, logits_input, token):
        native.check_logits_dtype(outs, "losses")
        native.require_cuda(outs, targets, weights)
        ctx.token = token
        outs = outs if outs.is_contiguous() else outs.contiguous()
        targets = _plane_contiguous(targets)
        B, K = outs.shape[0], outs.shape[1]
        n_pix = outs[0, 0].numel()
        if targets.shape[0] != B or targets.shape[1] != K or targets[0, 0].numel() != n_pix:
            raise native.NativeError("prediction / target shape mismatch: %s vs %s" % (tuple(outs.shape), tuple(targets.shape)))
        if weights.numel() != K:
            raise ValueError("class_weight has %d entries for %d classes" % (weights.numel(), K))
        dev, st = outs.device, stream_of(outs)
        stats = torch.empty((B, K, native.NSTAT), dtype=torch.float64, device=dev)
        out4 = torch.empty((4,), dtype=torch.float32, device=dev)
        coef = torch.empty((B, K, 3), dtype=torch.float32, device=dev)
        call("rhseg_loss_stats", ptr(outs), ptr(targets), targets.stride(0), targets.stride(1), B, K, n_pix,
             (1 if logits_input else 0) | native.logits_flag(outs), ptr(stats), st)
        call("rhseg_loss_finalize", ptr(stats), ptr(weights), B, K, float(smooth), ptr(out4), ptr(coef), st)
        ctx.save_for_backward(outs, targets, coef)
        ctx.logits_input = logits_input
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(stats)
        return out4[0], out4[1], out4[2:4], stats

    @staticmethod
    def backward(ctx, g_ce, g_dice, _g_counts, _g_stats):
        outs, targets, coef = ctx.saved_tensors
        ctx.token[0] = False  # this node has run backward: a memoised result must not be handed out again (its graph is freed)
        if g_ce is None and g_dice is None:
            return None, None, None, None, None, None
        B, K = outs.shape[0], outs.shape[1]
        n_pix = outs[0, 0].numel()

        def scalar(g):
            if g is None:
                return None
            g = g.reshape(1)
            return g if g.dtype == torch.float32 else g.float()

        g_ce, g_dice = scalar(g_ce), scalar(g_dice)
        dz = torch.empty_like(outs)  # bf16 predictions get a bf16 gradient
        call("rhseg_loss_bwd", ptr(outs), ptr(targets), targets.stride(0), targets.stride(1), ptr(coef),
             ptr(g_ce), ptr(g_dice), B, K, n_pix, (1 if ctx.logits_input else 0) | native.logits_flag(outs), ptr(dz),
             stream_of(outs))
        return dz, None, None, None, None, None


class LevelLoss:
    """Result of one fused level-loss evaluation."""
    __slots__ = ("ce", "dice", "counts", "stats")

    def __init__(self, ce, dice, counts, stats):
        self.ce, self.dice, self.counts, self.stats = ce, dice, counts, stats

    def dice_or_none(self):
        """Reference convention (losses.py:66): None when every sample's dice was NaN.  Needs one
        host read; skipped (tensor returned) while a CUDA graph is being captured."""
        if torch.cuda.is_current_stream_capturing():
            return self.dice
        return self.dice if float(self.counts[0].item()) > 0 else None


# (outs_ref, outs_version, targets_ref, targets_version, key, result, token).  token[0] turns False once the node has run
# backward (a second consumer then gets a fresh node instead of a freed graph).  Results carry autograd
# history, so the memo is kept tiny: the reference calls CE then Dice on the same tensors
# back to back (train.py:136-137) and one or two live entries cover that.
_MEMO = []
_MEMO_MAX = 2


def clear_memo():
    """Drops the memoised level losses (and the autograd history they keep alive)."""
    del _MEMO[:]



def level_loss(outs, targets, class_weight, smooth: Optional[float], logits_input: bool) -> LevelLoss:
    """CE + Dice of one level.  smooth=None (the CE module) accepts a memoised result computed
    with any smooth; a miss then computes with smooth=0."""
    grad = torch.is_grad_enabled() and outs.requires_grad
    wkey = tuple(float(w) for w in class_weight) if class_weight is not None else None
    for i in range(len(_MEMO) - 1, -1, -1):
        o_ref, o_ver, t_ref, t_ver, key, res, token = _MEMO[i]
        o, t = o_ref(), t_ref()
        if o is None or t is None or not token[0]:
            del _MEMO[i]
            continue
        if o is outs and t is targets and o_ver == outs._version and t_ver == targets._version \
                and key[0] == wkey and key[1] == bool(logits_input) and key[2] == grad \
                and (smooth is None or key[3] == float(smooth)):
            return res
    w = weight_tensor(class_weight, outs.device)
    sm = 0.0 if smooth is None else float(smooth)
    token = [True]
    with native.device_guard(outs):
        ce, dice, counts, stats = _LevelLossFn.apply(outs, targets, w, sm, bool(logits_input), token)
    res = LevelLoss(ce, dice, counts, stats)
    _MEMO.append((weakref.ref(outs), outs._version, weakref.ref(targets), targets._version,
                  (wkey, bool(logits_input), grad, sm), res, token))
    if len(_MEMO) > _MEMO_MAX:
        del _MEMO[0]
    return res


class _ConsistencyFn(torch.autograd.Function):
    """sum over groups of sum_{b,n} |sum_children P_c - P_parent| for one level pair."""

    @staticmethod
    def forward(ctx, cur, prev, table, n_groups):
        native.require_cuda(cur, prev)
        cur = cur if cur.is_contiguous() else cur.contiguous()
        prev = prev if prev.is_contiguous() else prev.contiguous()
        B, K = cur.shape[0], cur.shape[1]
        n_pix = cur[0, 0].numel()
        sums = torch.empty((native.MAX_K,), dtype=torch.float64, device=cur.device)
        call("rhseg_consistency_sums", ptr(cur), ptr(prev), ptr(table), B, K, prev.shape[1], n_pix, ptr(sums),
             stream_of(cur))
        ctx.save_for_backward(cur, prev, table)
        return sums[:n_groups]

    @staticmethod
    def backward(ctx, g):
        # Never exercised by the reference's training loop (its probabilities are constants there,
        # SURVEY.md F5); provided for completeness with elementwise device ops.
        cur, prev, table = ctx.saved_tensors
        tb = table.tolist()
        G = tb[1]
        d_cur, d_prev = torch.zeros_like(cur), torch.zeros_like(prev)
        for gi in range(G):
            s0, ln, par = tb[4 + 2 * native.MAX_K + gi], tb[4 + 3 * native.MAX_K + gi], tb[4 + 4 * native.MAX_K + gi]
            sign = torch.sign(cur[:, s0:s0 + ln].sum(1, keepdim=True) - prev[:, par:par + 1]) * g[gi].to(cur.dtype)
            d_cur[:, s0:s0 + ln] += sign
            d_prev[:, par:par + 1] -= sign
        return d_cur, d_prev, None, None


def consistency_loss(probs_per_level, levels, parent_of, reduction="mean"):
    """hierarchical_consistency_loss (Metrics/losses.py:150-177)."""
    if probs_per_level is None or levels is None or parent_of is None:
        return probs_per_level[0].sum() * 0 if probs_per_level else 0.0
    tree = tree_from_levels(levels, parent_of)
    dev = probs_per_level[0].device
    tables = tree.device_tables(dev)
    total, count = None, 0
    for L in range(1, tree.num_levels):
        G = tree.group_count(L)
        if G == 0:
            continue
        cur, prev = probs_per_level[L], probs_per_level[L - 1]
        with native.device_guard(cur):
            sums = _ConsistencyFn.apply(cur.float(), prev.float(), tables[L], G)
        if reduction == "mean":
            sums = sums / float(prev.shape[0] * prev[0, 0].numel())
        part = sums.sum()
        total = part if total is None else total + part
        count += G
    if count == 0:
        return probs_per_level[0].sum() * 0
    return (total / count).to(torch.float32)
