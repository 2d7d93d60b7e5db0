"""Fused training step of the restrictive-hierarchy path: head forward, train-path prediction,
confusion-matrix metrics, CE + Dice + consistency loss and the complete backward, as ONE
autograd node over the sm_100a kernels.

It computes exactly what the body of the reference's train_epoch computes between the donor
backbone and the optimiser (train.py:201-241: model head -> argmax/one-hot/mask glue ->
get_metrics -> get_loss -> backward), but
  * the one-hot prediction and eval-target tensors never exist (rhseg_level_eval reads logits
    and ternary targets once per level and emits statistics, confusion matrix, consistency sums
    and a uint8 index map),
  * the per-level loss gradient, the activation backward and (HRNet) the upsample adjoint are one
    kernel (rhseg_head_dz_*_fused), so no gradient tensor exists at output resolution for HRNet,
  * nothing synchronises with the host: all scalars come back in one small device tensor.
The drop-in modules (Models/, Metrics/) give the same numbers through the reference's own call
sequence; this is the additive fast path (INTEGRATION.md, "fused step").
"""
import ctypes
from typing import List, Optional, Sequence, Tuple

import torch

from . import native
from .head import backward_buffers, forward_levels, level_weight_backward
from .native import call, ptr, stream_of
from .tree_tables import ClassTree

_I32 = ctypes.c_int32


def widen_targets(target: torch.Tensor) -> torch.Tensor:
    """fp32 view of the wide ternary target tensor.  int8 targets (the dataset's {1, 0, -1}; a quarter of the bytes over
    PCIe) are widened by one kernel (rhseg_targets_i8_to_f32); other dtypes go through torch."""
    if target.dtype == torch.float32:
        return target
    if target.dtype == torch.int8 and target.is_contiguous() and target.data_ptr() % 16 == 0:
        out = torch.empty(target.shape, dtype=torch.float32, device=target.device)
        call("rhseg_targets_i8_to_f32", ptr(target), target.numel(), ptr(out), stream_of(target))
        return out
    return target.float()


class StepOutput:
    """Everything one training step reports, still on the device (no host sync)."""
    __slots__ = ("loss", "scalars", "level_ce", "level_dice", "consistency", "confusion", "ratios", "probs", "logits",
                 "summary", "exchange", "global_summary")

    def __init__(self, loss, scalars, confusion, ratios, probs, logits, n, summary=None, exchange=None, global_summary=None):
        self.summary = summary                 # fp64 additive per-rank summary for dist.all_reduce_summary
        self.exchange = exchange               # summary + `exchange_tail` free fp64 slots behind it (dist.pack_exchange)
        self.global_summary = global_summary   # data-parallel steps: SUM over ranks of `summary` (dist.unpack_global reads it)
        self.loss = loss                       # 0-dim, differentiable
        self.scalars = scalars                 # [2 + 4*n] fp32: total, consistency, then (ce, dice, n_dice, n_ce) per level
        self.consistency = scalars[1]
        self.level_ce = [scalars[2 + 4 * L] for L in range(n)]
        self.level_dice = [scalars[3 + 4 * L] for L in range(n)]
        self.confusion = confusion             # per level int64 [nc,nc]
        self.ratios = ratios                   # per level fp32 [5,nc] (rows: dice, iou, accuracy, precision, recall)
        self.probs, self.logits = probs, logits


def _eval_layout(tree: ClassTree, B: int):
    """Word offsets (8-byte words) of each level's [stats | consistency sums | confusion] block."""
    offs, off = [], 0
    for L, K in enumerate(tree.head_channels):
        nc = K + 1 if L > 0 else K
        offs.append((off, off + B * K * native.NSTAT, off + B * K * native.NSTAT + native.MAX_K, nc))
        off += B * K * native.NSTAT + native.MAX_K + nc * nc
    return offs, off


def _step_target(tree: ClassTree, target: torch.Tensor):
    """The wide ternary target as the evaluation kernels read it (fp32, contiguous H*W planes) and each level's first
    channel in it."""
    native.require_cuda(target)
    target = widen_targets(target)
    if target.dim() != 4 or target.shape[1] != sum(tree.head_channels):
        raise native.NativeError("target must be [B, sum(K_L), H, W] with sum(K_L) = %d, got %s"
                                 % (sum(tree.head_channels), tuple(target.shape)))
    if not (target.stride(3) == 1 and target.stride(2) == target.shape[3]):
        target = target.contiguous()
    ch_off = [0]
    for k in tree.head_channels:
        ch_off.append(ch_off[-1] + k)
    return target, ch_off


def _check_eval_dims(target, dims):
    if dims[0] != target.shape[0] or (dims[4], dims[5]) != tuple(target.shape[2:]):
        raise native.NativeError("target %s does not match the head output [%d, *, %d, %d]"
                                 % (tuple(target.shape), dims[0], dims[4], dims[5]))


def _finalize(tree: ClassTree, ws, offs, weights_all, smooth, B, n_pix, n_active, xchg_tail, st):
    """rhseg_step_finalize over the levels' evaluation words: (scalars + ratios, backward coefficients, summary with
    `xchg_tail` free slots behind it, per-level confusion views, per-level ratio views)."""
    n = tree.num_levels
    dev = ws.device
    n_ratio = sum(5 * o[3] for o in offs)
    scal_all = torch.empty((2 + 4 * n + n_ratio,), dtype=torch.float32, device=dev)
    coef_all = torch.empty((B * sum(tree.head_channels) * 3,), dtype=torch.float32, device=dev)
    # [summary | xchg_tail slots for the parameter gradients]: the data-parallel exchange buffer
    summary = torch.empty((2 + 4 * n + sum(o[3] * o[3] for o in offs) + int(xchg_tail),), dtype=torch.float64, device=dev)
    Ks = (_I32 * n)(*tree.head_channels)
    Gs = (_I32 * n)(*[tree.group_count(L) for L in range(n)])
    call("rhseg_step_finalize", ptr(ws), ptr(weights_all), B, n, Ks, Gs, float(smooth), n_pix, (1 << n_active) - 1,
         ptr(scal_all), ptr(coef_all), ptr(summary), st)
    conf, ratios, r_off = [], [], 2 + 4 * n
    for L in range(n):
        nc = offs[L][3]
        conf.append(ws[offs[L][2]:offs[L][2] + nc * nc].view(torch.int64).view(nc, nc))
        ratios.append(scal_all[r_off:r_off + 5 * nc].view(5, nc))
        r_off += 5 * nc
    return scal_all, coef_all, summary, conf, ratios


def _n_active(n, level_cap):
    return n if level_cap is None else max(1, min(n, int(level_cap) + 1))  # train.py:121-126


class _FusedStepFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, tree: ClassTree, out_size, weights_all, smooth, xchg_tail, level_cap, dp, target, *tensors):
        n = tree.num_levels
        n_active = _n_active(n, level_cap)
        target, ch_off = _step_target(tree, target)
        dev = target.device
        B = target.shape[0]
        t_bs, t_cs = target.stride(0), target.stride(1)
        esz = target.element_size()
        offs, words = _eval_layout(tree, B)
        idx_maps = [torch.empty((B,) + tuple(target.shape[2:]), dtype=torch.uint8, device=dev) if L < n - 1 else None
                    for L in range(n)]

        def evaluate(L, dims, ws):  # ws: the zeroed statistics workspace (part of the forward's single fill)
            _check_eval_dims(target, dims)
            return (target.data_ptr() + ch_off[L] * t_cs * esz, t_bs, t_cs,
                    target.data_ptr() + ch_off[L - 1] * t_cs * esz if L > 0 else None,
                    ptr(idx_maps[L - 1]) if L > 0 else None, ws.data_ptr() + offs[L][0] * 8, ptr(idx_maps[L]))

        grad = any(ctx.needs_input_grad)  # grad mode is off inside forward(): ask autograd
        r = forward_levels(tree, out_size, tensors, evaluate, zero_words=words, with_backward=grad)
        ctx.bwd = r["bwd"]
        ws = r["workspace"]
        B, C, Hf, Wf, H, W = r["dims"]
        st = stream_of(r["feats"][0])
        scal_all, coef_all, summary, conf, ratios = _finalize(tree, ws, offs, weights_all, smooth, B, H * W, n_active,
                                                              xchg_tail, st)
        scalars = scal_all[:2 + 4 * n]
        # data-parallel: the summary is summed over ranks BETWEEN forward and backward (a few hundred bytes), because the
        # exact Dice gradient needs the global count of valid samples (dist.py, rhseg_dp_grad_scales)
        n_summary = summary.numel() - int(xchg_tail)
        ctx.dp = None
        gsum = summary[:0]
        if dp is not None:
            reduce_fn, world = dp
            gsum = reduce_fn(summary[:n_summary])
            if gsum.data_ptr() == summary.data_ptr():
                raise native.NativeError("the data-parallel summary reduction must not overwrite the local summary")
            ctx.dp = (summary, gsum, int(world))
        ctx.n_active = n_active
        ctx.tree, ctx.dims, ctx.upsampled = tree, r["dims"], r["upsampled"]
        ctx.t_meta = (t_bs, t_cs, ch_off, esz)
        ctx.save_for_backward(target, coef_all, *r["feats"], *r["head_w"], *r["film_w"], *r["logits"], *r["probs"],
                              *r["psums"], *r["eff_ws"], *[g for g in r["gbs"] if g is not None])
        ctx.set_materialize_grads(False)
        outs = (scalars[0], scalars) + tuple(conf) + tuple(ratios) + tuple(r["probs"]) + tuple(r["logits"]) + (summary, gsum)
        ctx.mark_non_differentiable(*outs[1:])
        return outs

    @staticmethod
    def backward(ctx, g_total, *_unused):
        tree = ctx.tree
        n = tree.num_levels
        B, C, Hf, Wf, H, W = ctx.dims
        sv = ctx.saved_tensors
        target, coef_all = sv[0], sv[1]
        sv = sv[2:]
        feats, head_w, film_w = sv[0:n], sv[n:2 * n], sv[2 * n:3 * n - 1]
        o = 3 * n - 1
        logits, probs, psums, eff_ws = sv[o:o + n], sv[o + n:o + 2 * n], sv[o + 2 * n:o + 3 * n], sv[o + 3 * n:o + 4 * n]
        gbs = [None] + list(sv[o + 4 * n:o + 5 * n - 1])
        t_bs, t_cs, ch_off, esz = ctx.t_meta
        n_grads = 5 * n - 2
        if g_total is None:
            return (None,) * (8 + n_grads)
        dev = feats[0].device
        st = stream_of(feats[0])
        tables = tree.device_tables(dev)
        n_pix = H * W
        g = g_total.reshape(1)
        g = g if g.dtype == torch.float32 else g.float()
        # accumulators zeroed by the forward's single fill; a second backward over the same graph gets fresh ones
        bufs, ctx.bwd = ctx.bwd, None
        if bufs is None:
            bufs = backward_buffers(tree, B, C, dev, (Hf, Wf) if ctx.upsampled else None)
        d_feats: List[Optional[torch.Tensor]] = [None] * n
        d_hw: List[Optional[torch.Tensor]] = [None] * n
        d_hb: List[Optional[torch.Tensor]] = [None] * n
        d_fw: List[Optional[torch.Tensor]] = [None] * (n - 1)
        d_fb: List[Optional[torch.Tensor]] = [None] * (n - 1)
        g_uniform, dp_pix, pix_mask = None, None, 0
        coef_off = 0
        coef_offs = []
        for k in tree.head_channels:
            coef_offs.append(coef_off)
            coef_off += B * k * 3
        g_ptrs = [(ptr(g), ptr(g))] * n
        if ctx.dp is not None:  # per-level (g_ce, g_dice) = g * the factors that make DDP's mean over ranks exact
            local, gsum, world = ctx.dp
            scales = torch.empty((2 * n,), dtype=torch.float32, device=dev)
            call("rhseg_dp_grad_scales", ptr(local), ptr(gsum), n, world, ptr(g), ptr(scales), st)
            g_ptrs = [(scales.data_ptr() + 8 * L, scales.data_ptr() + 8 * L + 4) for L in range(n)]
        # levels above the curriculum cap take no part in the loss: nothing reaches their logits (train.py:125-126)
        for L in range(ctx.n_active - 1, -1, -1):
            K = tree.head_channels[L]
            K_prev = tree.head_channels[L - 1] if L > 0 else 0
            mode = tree.act_mode[L]
            dp_prev, prev_mask = None, 0
            if mode == native.ACT_GROUPED and (g_uniform is not None or dp_pix is not None):
                dp_prev = torch.zeros((B, K_prev, H, W), dtype=torch.float32, device=dev)
                for pname, _ in tree.child_groups[L - 1]:
                    prev_mask |= 1 << tree.levels[L - 1].index(pname)
            t_ptr = target.data_ptr() + ch_off[L] * t_cs * esz
            c_ptr = coef_all.data_ptr() + coef_offs[L] * 4
            if ctx.upsampled:
                dz = bufs[L]["dz"]  # zeroed together with the weight sums: the band kernel adds into it
                call("rhseg_head_dz_lowres_fused", ptr(logits[L]), t_ptr, t_bs, t_cs, c_ptr, g_ptrs[L][0], g_ptrs[L][1],
                     ptr(probs[L - 1]) if L > 0 else None, ptr(tables[L]), ptr(g_uniform), 1.0 / n_pix, ptr(dp_pix),
                     pix_mask, B, K, K_prev, Hf, Wf, H, W, mode | tree.group_hint(L), ptr(dz), ptr(dp_prev), None,
                     native.DZ_PREZEROED, st)
            else:
                dz = torch.empty((B, K, H, W), dtype=torch.float32, device=dev)
                # nothing but the loss reaches the last active level's logits: the kernel instance without activation code
                # (64 instead of 122 registers for a grouped K = 4 level) gives the same gradient
                mode_bwd = native.ACT_ZEROS if (g_uniform is None and dp_pix is None) else mode
                call("rhseg_head_dz_fullres_fused", ptr(logits[L]), t_ptr, t_bs, t_cs, c_ptr, g_ptrs[L][0], g_ptrs[L][1],
                     ptr(probs[L - 1]) if L > 0 else None, ptr(tables[L]), ptr(g_uniform), 1.0 / n_pix, ptr(dp_pix),
                     pix_mask, B, K, K_prev, n_pix, mode_bwd, ptr(dz), ptr(dp_prev), st)
            d_feats[L], d_hw[L], d_hb[L], fw_g, fb_g, g_prev = level_weight_backward(
                tree, L, ctx.dims, feats[L], dz, eff_ws[L], head_w[L], film_w[L - 1] if L > 0 else None, gbs[L],
                psums[L - 1] if L > 0 else None, bufs[L], ctx.needs_input_grad[8 + L], st)
            if L > 0:
                d_fw[L - 1], d_fb[L - 1] = fw_g, fb_g
            g_uniform, dp_pix, pix_mask = g_prev, dp_prev, prev_mask
        return (None,) * 8 + tuple(d_feats) + tuple(d_hw) + tuple(d_hb) + tuple(d_fw) + tuple(d_fb)


class FusedHierStep:
    """Callable fused training step for one class tree and one set of per-level class weights.

        step = FusedHierStep(tree_dict, level_weights)
        out = step(feats, head_w, head_b, film_w, film_b, target, out_size=None)
        out.loss.backward()            # or torch.autograd.grad(out.loss, ...)

    `target` is the wide ternary tensor [B, sum(K_L), H, W] of the dataset (train.py:181-193).
    """

    def __init__(self, hierarchy, level_weights: Sequence[Sequence[float]], smooth: float = 0.0):
        self.tree = hierarchy if isinstance(hierarchy, ClassTree) else ClassTree(hierarchy)
        if len(level_weights) != self.tree.num_levels:
            raise ValueError("level_weights needs one list per level")
        for L, w in enumerate(level_weights):
            if len(w) != self.tree.head_channels[L]:
                raise ValueError("level %d has %d classes but %d weights" % (L, self.tree.head_channels[L], len(w)))
        self._weights_host = [float(x) for w in level_weights for x in w]
        self._weights = {}
        self.smooth = float(smooth)
        # free fp64 slots allocated behind StepOutput.summary (data-parallel jobs: set it to the number of
        # parameter-gradient elements that ride in the step's all-reduce, see dist.pack_exchange)
        self.exchange_tail = 0
        self._dp = None
        if self.tree.num_levels > 8:
            raise native.NativeError("fused step supports trees up to 8 levels deep")

    def weights(self, device):
        key = str(device)
        if key not in self._weights:
            self._weights[key] = torch.tensor(self._weights_host, dtype=torch.float32).to(device)
        return self._weights[key]

    def data_parallel(self, reduce_fn, world: int):
        """Batch-sharded training (one process per GPU): `reduce_fn(summary) -> new fp64 tensor` = SUM over ranks of the
        step summary (e.g. `lambda s: px.all_reduce(s)` with a dist.PeerExchange, or a clone + torch.distributed.all_reduce).
        It runs between forward and backward; the backward then scales each level's CE / Dice gradient so that DDP's mean
        over ranks equals the single-process gradient on the concatenated batch, also when the ranks hold different
        numbers of dice-valid samples (Metrics/losses.py:64-66).  reduce_fn=None switches it off."""
        self._dp = None if reduce_fn is None else (reduce_fn, int(world))

    def __call__(self, feats, head_w, head_b, film_w, film_b, target, out_size: Optional[Tuple[int, int]] = None,
                 level_cap: Optional[int] = None) -> StepOutput:
        """level_cap: the reference's level-pretrain curriculum (train.get_loss, train.py:121-126): only levels
        L <= level_cap = min(n-1, cur_epoch // pretrain_epoch) enter the loss and receive gradients; every level's
        CE / Dice value, metrics and the consistency term are still reported.  None = all levels."""
        n = self.tree.num_levels
        if not (len(feats) == len(head_w) == len(head_b) == n and len(film_w) == len(film_b) == n - 1):
            raise native.NativeError("expected %d levels of features/heads and %d FiLMs" % (n, n - 1))
        with torch.cuda.device(feats[0].device):  # kernels launch on the tensors' device, whatever the current one is
            outs = _FusedStepFn.apply(self.tree, out_size, self.weights(feats[0].device), self.smooth, self.exchange_tail,
                                      level_cap, self._dp, target, *feats, *head_w, *head_b, *film_w, *film_b)
        xbuf, gsum = outs[2 + 4 * n], outs[3 + 4 * n]
        return StepOutput(outs[0], outs[1], list(outs[2:2 + n]), list(outs[2 + n:2 + 2 * n]),
                          list(outs[2 + 2 * n:2 + 3 * n]), list(outs[2 + 3 * n:2 + 4 * n]), n,
                          xbuf[:xbuf.numel() - self.exchange_tail], xbuf, gsum if gsum.numel() else None)

    def validate(self, feats, head_w, head_b, film_w, film_b, target, out_size: Optional[Tuple[int, int]] = None,
                 level_cap: Optional[int] = None, keep_outputs: bool = False) -> StepOutput:
        """Validation pass of one batch: the numbers the reference's test() reports (train.py:282-393, evaluation at
        :324-339), which are not those of the training step (DESIGN.md 3.9):
          * metrics: ProcessClasses over the COMPOSED probabilities against the raw ternary targets (the step: argmax
            of softmax(z) over all K logits, one-hot masked where the target is -1, against -1 -> 0 targets);
          * consistency: on the real probabilities (the step: on the masked one-hots);
          * CE and Dice: the same as the step's.
        Arguments, level_cap, int8 targets and bf16 / channels-last features as in __call__.  Never records autograd,
        whatever the grad mode (out.loss.requires_grad is False), allocates no backward buffers and never synchronises
        with the host, so it can be captured in a CUDA graph.  keep_outputs=False: out.probs / out.logits are None and
        only the previous level's probabilities stay alive while a level runs; True returns every level's.
        out.summary is additive over batches and ranks: dist.unpack_global(sum of the summaries) gives the epoch's
        numbers.  With data_parallel set, out.global_summary = reduce_fn(out.summary)."""
        n = self.tree.num_levels
        if not (len(feats) == len(head_w) == len(head_b) == n and len(film_w) == len(film_b) == n - 1):
            raise native.NativeError("expected %d levels of features/heads and %d FiLMs" % (n, n - 1))
        native.require_cuda(feats[0], target)
        with torch.no_grad(), torch.cuda.device(feats[0].device):
            tree = self.tree
            target, ch_off = _step_target(tree, target)
            B = target.shape[0]
            t_bs, t_cs, esz = target.stride(0), target.stride(1), target.element_size()
            offs, words = _eval_layout(tree, B)

            def evaluate(L, dims, ws):
                _check_eval_dims(target, dims)
                return target.data_ptr() + ch_off[L] * t_cs * esz, t_bs, t_cs, ws.data_ptr() + offs[L][0] * 8

            r = forward_levels(tree, out_size, (*feats, *head_w, *head_b, *film_w, *film_b), evaluate, zero_words=words,
                               composed=True, keep_outputs=keep_outputs)
            B, C, Hf, Wf, H, W = r["dims"]
            scal_all, _, summary, conf, ratios = _finalize(tree, r["workspace"], offs, self.weights(target.device),
                                                           self.smooth, B, H * W, _n_active(n, level_cap), 0,
                                                           stream_of(r["feats"][0]))
            gsum = None
            if self._dp is not None:
                gsum = self._dp[0](summary)
                if gsum.data_ptr() == summary.data_ptr():
                    raise native.NativeError("the data-parallel summary reduction must not overwrite the local summary")
        probs, logits = (r["probs"], r["logits"]) if keep_outputs else ([None] * n, [None] * n)
        return StepOutput(scal_all[0], scal_all[:2 + 4 * n], conf, ratios, probs, logits, n, summary, summary, gsum)


class _FusedFlatFn(torch.autograd.Function):
    """Flat model (model_type 0; Models/models.py:258-261, :754-757): weighted CE + Dice on the logits of ONE level of
    leaf classes, the train-path prediction and the confusion-matrix metrics, in three launches: rhseg_level_eval
    (statistics + bit-exact argmax(softmax) + confusion, one pass over logits and targets), rhseg_step_finalize,
    and rhseg_head_dz_fullres_fused in the backward (closed-form gradient, one pass).  bf16 logits (a flat head run under
    bf16 autocast) are read as such (RHSEG_LOGITS_BF16): the results are those of the fp32 step on logits.float(), and
    the gradient comes back as bf16, rounded once."""

    @staticmethod
    def forward(ctx, tree: ClassTree, weights, smooth, logits, target):
        native.require_cuda(logits, target)
        z = logits if logits.is_contiguous() else logits.contiguous()
        t = widen_targets(target)
        if not (t.stride(3) == 1 and t.stride(2) == t.shape[3]):
            t = t.contiguous()
        B, K, H, W = z.shape
        if tuple(t.shape) != tuple(z.shape) or K != tree.head_channels[0]:
            raise native.NativeError("flat step: logits %s / targets %s / %d classes do not match"
                                     % (tuple(z.shape), tuple(t.shape), tree.head_channels[0]))
        dev, st = z.device, stream_of(z)
        n_pix = H * W
        offs, words = _eval_layout(tree, B)
        ws = torch.zeros((words,), dtype=torch.float64, device=dev)
        tables = tree.device_tables(dev)
        call("rhseg_level_eval", ptr(z), ptr(t), t.stride(0), t.stride(1), None, 0, 0, None, ptr(tables[0]), B, K, n_pix, 0,
             ptr(ws), None, native.EVAL_PREZEROED | native.logits_flag(z), st)
        scal_all = torch.empty((2 + 4 + 5 * K,), dtype=torch.float32, device=dev)
        coef = torch.empty((B * K * 3,), dtype=torch.float32, device=dev)
        summary = torch.empty((2 + 4 + K * K,), dtype=torch.float64, device=dev)
        Ks, Gs = (_I32 * 1)(K), (_I32 * 1)(0)
        call("rhseg_step_finalize", ptr(ws), ptr(weights), B, 1, Ks, Gs, float(smooth), n_pix, 1, ptr(scal_all), ptr(coef),
             ptr(summary), st)
        conf = ws[offs[0][2]:offs[0][2] + K * K].view(torch.int64).view(K, K)
        ratios = scal_all[6:6 + 5 * K].view(5, K)
        ctx.save_for_backward(z, t, coef, tables[0])
        ctx.set_materialize_grads(False)
        outs = (scal_all[0], scal_all[:6], conf, ratios, summary)
        ctx.mark_non_differentiable(*outs[1:])
        return outs

    @staticmethod
    def backward(ctx, g_total, *_unused):
        if g_total is None:
            return None, None, None, None, None
        z, t, coef, table = ctx.saved_tensors
        B, K, H, W = z.shape
        g = g_total.reshape(1)
        g = g if g.dtype == torch.float32 else g.float()
        dz = torch.empty_like(z)
        call("rhseg_head_dz_fullres_fused", ptr(z), ptr(t), t.stride(0), t.stride(1), ptr(coef), ptr(g), ptr(g), None, ptr(table),
             None, 1.0 / (H * W), None, 0, B, K, 0, H * W, native.ACT_ZEROS | native.logits_flag(z), ptr(dz), None,
             stream_of(z))  # no activation path:
        # nothing but the loss reaches the flat logits (the instance without activation code: 108 vs 138 registers at K = 7)
        return None, None, None, dz, None


class FusedFlatStep:
    """Loss + metrics of the flat baseline (BASELINE.json configs[3]: model_type 0, 7 leaf classes, README.md:79 weights):

        step = FusedFlatStep(class_names_or_count, class_weight)
        out = step(logits, target)          # logits [B,K,H,W] from the donor's flat head, target {0,1} one-hots
        out.loss.backward()                 # d(CE + Dice)/d logits

    Same numbers as CrossEntropyLoss + SoftDiceLoss (Metrics/losses.py) and the five metric wrappers called the way
    train.py calls them for a flat model, without one-hot tensors and without a host sync."""

    def __init__(self, classes, class_weight: Sequence[float], smooth: float = 0.0):
        names = ["c%d" % i for i in range(classes)] if isinstance(classes, int) else list(classes)
        if len(class_weight) != len(names):
            raise ValueError("%d classes but %d weights" % (len(names), len(class_weight)))
        self.tree = ClassTree({n: {} for n in names})
        self._weights_host = [float(x) for x in class_weight]
        self._weights = {}
        self.smooth = float(smooth)

    def __call__(self, logits, target) -> StepOutput:
        """logits: float32, or bfloat16 (a flat head under bf16 autocast: the results are the fp32 step's on
        logits.float(), and the gradient reaching the logits is bf16)."""
        native.check_logits_dtype(logits, "flat step")
        key = str(logits.device)
        if key not in self._weights:
            self._weights[key] = torch.tensor(self._weights_host, dtype=torch.float32).to(logits.device)
        with torch.cuda.device(logits.device):
            loss, scalars, conf, ratios, summary = _FusedFlatFn.apply(self.tree, self._weights[key], self.smooth, logits, target)
        return StepOutput(loss, scalars, [conf], [ratios], [None], [logits], 1, summary, summary)
