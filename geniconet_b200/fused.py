"""Fused execution of the residual encoder / decoder bodies of models.py (SURVEY 8f rank 1).

The module-by-module path (ico_conv.py + torch BatchNorm2d / ReLU / add, exactly what the unmodified models.py runs) moves every
conv output through five torch kernels before the next conv sees it.  Here a whole chain of

    stem   IcoConvS2S(3 -> C) + BatchNorm2d + ReLU                                   (models.py:104-111)
    block  BasicIcoS2SDownBlock / BasicIcoS2SUpBlock                                 (models.py:22-62)

runs inside ONE autograd Function whose internal activations exist only as the bf16 operand copies the tcgen05 kernels gather
from (plus the fp32 conv outputs BatchNorm needs):

  * the two sibling convolutions of a block (conv00 / conv10 read the same input) are one GEMM with concatenated output
    channels -- forward, wgrad and (concatenated along K, which also adds the two input gradients for free) dgrad;
  * BatchNorm statistics, normalise + ReLU + residual add + bf16 cast are gin_bn_stats / gin_bn_act_fwd, their backward
    gin_bn_act_bwd writes the bf16 gradient copy dgrad and wgrad read (include/geniconet_b200.h);
  * an Up block upsamples once (upsample00 / upsample10 are the same parameter-free map), from the fp32 coarse map straight
    into the bf16 operand copy of the fine level.

Parameters stay where models.py puts them (conv00.weight, icobn00.weight, ...), so state dicts are unchanged; BatchNorm running
statistics are updated as torch does.  With grad disabled, infer_chain runs the same chains forward-only (eval mode: BatchNorm in
the conv epilogue, DESIGN "Inference").  Eval mode with grad enabled runs run_frozen_chain (opt-in, DESIGN "Frozen BatchNorm"):
the training chain's forward kernels with the running statistics, nothing updated, and a backward of one streaming pass per
BatchNorm (gin_bn_eval_bwd / _pair) that computes weight gradients only for weights that need them.
In train mode a conv bias that feeds a BatchNorm has a mathematically zero gradient and the training chain returns exactly zero
for it; in eval mode its gradient is scale * sum(g), which the frozen chain returns.
A chain of SyncBatchNorm (torch.nn.SyncBatchNorm.convert_sync_batchnorm) runs the same chains; in training, when torch would
synchronise, every BatchNorm reduction all-gathers one fp64 record per rank and sums the records in rank order (sync_group,
_exchange; DESIGN "Synchronised BatchNorm").
"""
import torch

from . import _lib
from .ico_conv import IcoConvS2S, get_plan, _stream, pixel_strides, as_channels_last, cast_bf16

L = _lib.lib


def _P(level):
    return 10 * 4 ** level


def _is_block(m):
    return hasattr(m, 'conv00') and hasattr(m, 'icobn10')


# The BatchNorms a chain runs.  A SyncBatchNorm in eval mode is a plain BatchNorm; in train mode the training chain synchronises
# its statistics over its process group (sync_group).
_BN = (torch.nn.BatchNorm2d, torch.nn.SyncBatchNorm)


def chain_supported(mods):
    """True when `mods` is [IcoConvS2S(3->C), BatchNorm, ReLU]? + residual blocks with tensor-core channel widths, and its BatchNorms
    are all BatchNorm2d or all SyncBatchNorm on one process group."""
    mods = list(mods)
    i = 0
    if len(mods) >= 3 and isinstance(mods[0], IcoConvS2S) and isinstance(mods[1], _BN) and isinstance(mods[2], torch.nn.ReLU):
        if mods[0].in_features != 3 or mods[0].stride != 1 or mods[0].out_features % 64 or mods[0].bias is None:
            return False
        i = 3
    if i == len(mods):
        return False
    if i == 3 and _is_block(mods[3]) and not mods[3]._down:
        return False                                  # an Up block needs the fp32 map of its input, the stem keeps only the bf16 copy
    for m in mods[i:]:
        if not _is_block(m):
            return False
        for c in (m.conv00, m.conv01, m.conv10):
            if c.in_features % 64 or c.out_features % 64 or c.bias is None or 256 % (c.out_features // 8):
                return False
        for b in (m.icobn00, m.icobn01, m.icobn10):
            if not isinstance(b, _BN) or not b.affine or not b.track_running_stats or b.momentum is None:
                return False
    bns = [bn for bn, _ in eval_pairs(mods)]
    return len({isinstance(bn, torch.nn.SyncBatchNorm) for bn in bns}) == 1 and len({id(getattr(bn, 'process_group', None)) for bn in bns}) == 1


def sync_group(mods):
    """(process group, world size, rank in it) over which the training chain `mods` (see chain_supported) synchronises its BatchNorm
    statistics, or None when it does not: BatchNorm2d, or SyncBatchNorm that torch would not synchronise either (torch.distributed
    not initialised, or a group of one rank)."""
    bn = mods[1] if isinstance(mods[0], IcoConvS2S) else mods[0].icobn00
    if not isinstance(bn, torch.nn.SyncBatchNorm):
        return None
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return None
    world = dist.get_world_size(bn.process_group)
    return (bn.process_group, world, dist.get_rank(bn.process_group)) if world > 1 else None


def chain_params(mods):
    out = []
    for m in mods:
        if isinstance(m, IcoConvS2S):
            out += [m.weight, m.bias]
        elif isinstance(m, _BN):
            out += [m.weight, m.bias]
        elif _is_block(m):
            for c, b in ((m.conv00, m.icobn00), (m.conv01, m.icobn01), (m.conv10, m.icobn10)):
                out += [c.weight, c.bias, b.weight, b.bias]
    return out


# ------------------------------------------------------------------------------------------------ thin wrappers over the C ABI
def _empty(n, dtype, dev):
    return torch.empty(n, dtype=dtype, device=dev)


def _pack(w, cin, cout):
    packed = _empty(L.gin_hexconv_packed_bytes(cin, cout), torch.uint8, w.device)
    _lib.check(L.gin_hexconv_pack_weights(w.data_ptr(), packed.data_ptr(), cin, cout, _stream()), 'gin_hexconv_pack_weights')
    return packed


def _pack_many(jobs):
    """jobs: list of (w0, w1 or None, cin) -> list of packed blobs (16-bit tile images only), ONE launch for all of them."""
    import ctypes
    n = len(jobs)
    if n == 0:
        return []
    if n > 24:
        return _pack_many(jobs[:24]) + _pack_many(jobs[24:])
    dev = jobs[0][0].device
    outs = [_empty(L.gin_hexconv_packed_bytes(cin, w0.shape[0] + (w1.shape[0] if w1 is not None else 0)), torch.uint8, dev) for w0, w1, cin in jobs]
    P, I = ctypes.c_void_p * n, ctypes.c_int * n
    w0s = P(*[w0.data_ptr() for w0, _, _ in jobs])
    w1s = P(*[(w1.data_ptr() if w1 is not None else None) for _, w1, _ in jobs])
    c0 = I(*[w0.shape[0] for w0, _, _ in jobs])
    c1 = I(*[(w1.shape[0] if w1 is not None else 0) for _, w1, _ in jobs])
    pk = P(*[o.data_ptr() for o in outs])
    ci = I(*[cin for _, _, cin in jobs])
    _lib.check(L.gin_hexconv_pack_weights_bf16_multi(n, w0s, c0, w1s, c1, pk, ci, _stream()), 'gin_hexconv_pack_weights_bf16_multi')
    return outs


def _conv_fwd(plan, xb, packed, bias, B, cin, cout, p_out, bias1=None):
    """Returns (y fp32 [B*p_out][cout], per-CTA BatchNorm partial sums [nparts][2][cout] or None).  With `bias1` the output
    channels are two sibling convolutions side by side: `bias` belongs to the first half, `bias1` to the second."""
    import ctypes
    parts = _empty(L.gin_hexconv_stats_ws_bytes(cout) // 4, torch.float32, xb.device)
    n = ctypes.c_int(0)
    # The output is only ever read by the BatchNorm kernels: written as fp16 (GIN_Y_FP16=0: fp32) it costs half the bytes of its
    # one write and three reads; the statistics come from the fp32 accumulators either way.
    y = _empty((B * p_out, cout), torch.float16 if _Y16 else torch.float32, xb.device)
    rc = L.gin_hexconv_fwd_bf16_stats2(plan.host_ptr, plan.dev_ptr, xb.data_ptr(), packed.data_ptr(), bias.data_ptr(),
                                       bias1.data_ptr() if bias1 is not None else None, cout // 2 if bias1 is not None else 0,
                                       y.data_ptr(), 1 if _Y16 else 0, B, cin, cout, parts.data_ptr(), ctypes.addressof(n), _stream())
    if rc == 0:
        return y, ((parts, n.value) if n.value > 0 else None)
    if rc != _lib.ERR_UNSUPPORTED:
        _lib.check(rc, 'gin_hexconv_fwd_bf16_stats2')
    # a kernel generation without the second bias pointer / the fp16 epilogue
    y = _empty((B * p_out, cout), torch.float32, xb.device)
    if bias1 is not None:
        bias = torch.cat((bias, bias1), 0)
    _lib.check(L.gin_hexconv_fwd_bf16_stats(plan.host_ptr, plan.dev_ptr, xb.data_ptr(), packed.data_ptr(), bias.data_ptr(), y.data_ptr(), B, cin, cout,
                                            parts.data_ptr(), ctypes.addressof(n), _stream()), 'gin_hexconv_fwd_bf16_stats')
    return y, ((parts, n.value) if n.value > 0 else None)


def _conv_dgrad(plan, dyb, packed, B, cin, cout, p_in):
    dx = _empty((B * p_in, cin), torch.float32, dyb.device)
    _lib.check(L.gin_hexconv_dgrad_bf16(plan.host_ptr, plan.dev_ptr, dyb.data_ptr(), packed.data_ptr(), dx.data_ptr(), B, cin, cout, _stream()),
               'gin_hexconv_dgrad_bf16')
    return dx


def _conv_wgrad(plan, xb, dyb, B, cin, cout, out=None):
    """dW [cout][cin][7] (written into `out` when given: a data-parallel bucket slot)."""
    dW = out if out is not None else _empty((cout, cin, 7), torch.float32, xb.device)
    ws = _empty(L.gin_hexconv_wgrad_ws_bytes(cin, cout), torch.uint8, xb.device)
    _lib.check(L.gin_hexconv_wgrad_bf16(plan.host_ptr, plan.dev_ptr, xb.data_ptr(), dyb.data_ptr(), None, dW.data_ptr(), None, ws.data_ptr(),
                                        B, cin, cout, _stream()), 'gin_hexconv_wgrad_bf16')
    return dW


import os as _os
_Y16 = _os.environ.get('GIN_Y_FP16', '1') != '0'
_grad_sink = None
_grad_dest = None


def set_grad_sink(fn):
    """fn(list of (parameter, gradient)) is called from inside a chain's backward as soon as a block's gradients are enqueued
    (data-parallel training: geniconet_b200.dp.GradBuckets starts the all-reduce of a complete bucket right there); None
    removes it.  The chain still returns the same gradients to autograd afterwards."""
    global _grad_sink
    _grad_sink = fn


def set_grad_dest(fn):
    """fn(tuple of parameters) -> a contiguous fp32 tensor that IS the gradient storage of those parameters laid end to end (a
    slot of a data-parallel bucket), or None.  The chain's wgrad kernels then write straight into it (no bucket copy)."""
    global _grad_dest
    _grad_dest = fn


def weight_pairs(model):
    """The (conv00.weight, conv10.weight) pairs of every residual block: their gradients come out of ONE wgrad GEMM as one
    [2*Cout, Cin, 7] tensor, so a data-parallel bucket that keeps each pair adjacent can receive it in place."""
    return [(m.conv00.weight, m.conv10.weight) for m in model.modules() if _is_block(m)]


def _dest(params, shape):
    if _grad_dest is None:
        return None
    t = _grad_dest(params)
    return t.view(shape) if t is not None and t.numel() == int(torch.Size(shape).numel()) else None


def _exchange(rec, sync):
    """All-gather of this rank's fp64 record over sync = (process group, world, rank): [world][record], in rank order.  Every rank
    issues the chain's exchanges in the same order."""
    out = torch.empty(sync[1] * rec.numel(), dtype=torch.float64, device=rec.device)      # flat: gloo takes no other shape
    torch.distributed.all_gather_into_tensor(out, rec, group=sync[0])
    return out


def _bn_ptrs(bn, stat):
    """gin_bn_sync_stats_final's arguments of one BatchNorm; (None, ...) for the absent second one"""
    if bn is None:
        return [None, None, 0.0, 0.0, None, None, None, None]
    return [bn.weight.data_ptr(), bn.bias.data_ptr(), float(bn.eps), float(bn.momentum), bn.running_mean.data_ptr(), bn.running_var.data_ptr(),
            bn.num_batches_tracked.data_ptr(), stat.data_ptr()]


def _sync_stats(y, cols, ld, rows, C, parts, sync, targets):
    """Synchronised batch statistics of the BatchNorms `targets` = [(bn, stat)] (one, or a sibling pair) whose inputs are columns
    `cols` of y: this rank's record (from the epilogue partials, else from the fp32 map), one exchange, the final over every rank."""
    dev = y.device
    rec = _empty(L.gin_bn_sync_record_bytes(C, len(targets) - 1) // 8, torch.float64, dev)
    if parts is not None:
        _lib.check(L.gin_bn_sync_stats_total_from_parts(parts[0].data_ptr(), parts[1], ld, rows, C, cols[0], cols[1] if len(cols) > 1 else -1,
                                                        rec.data_ptr(), _stream()), 'gin_bn_sync_stats_total_from_parts')
    else:
        assert y.dtype == torch.float32, 'gin_bn_sync_stats_total reads fp32 maps (fp16 conv outputs always come with epilogue statistics)'
        ws = _empty(L.gin_bn_ws_bytes(C), torch.uint8, dev)
        for q, col in enumerate(cols):
            _lib.check(L.gin_bn_sync_stats_total(y.data_ptr() + 4 * col, ld, rows, C, rec.data_ptr() + 8 * q * (2 * C + 1), ws.data_ptr(), _stream()),
                       'gin_bn_sync_stats_total')
    recs = _exchange(rec, sync)
    (bnA, statA), (bnB, statB) = targets[0], (targets[1] if len(targets) > 1 else (None, None))
    _lib.check(L.gin_bn_sync_stats_final(recs.data_ptr(), sync[1], C, *_bn_ptrs(bnA, statA), *_bn_ptrs(bnB, statB), _stream()), 'gin_bn_sync_stats_final')


def _bn_stats(y, col0, ld, rows, C, bn, parts=None, sync=None):
    stat = _empty(4 * C, torch.float32, y.device)
    if sync is not None:
        _sync_stats(y, (col0,), ld, rows, C, parts, sync, [(bn, stat)])
        return stat
    if parts is not None:         # the conv epilogue already summed y and y^2 per CTA
        pbuf, n = parts
        _lib.check(L.gin_bn_stats_from_parts(pbuf.data_ptr() + 4 * col0, n, ld, rows, C, bn.weight.data_ptr(), bn.bias.data_ptr(), float(bn.eps),
                                             float(bn.momentum), bn.running_mean.data_ptr(), bn.running_var.data_ptr(),
                                             bn.num_batches_tracked.data_ptr(), stat.data_ptr(), _stream()), 'gin_bn_stats_from_parts')
        return stat
    assert y.dtype == torch.float32, 'gin_bn_stats reads fp32 maps (fp16 conv outputs always come with epilogue statistics)'
    ws = _empty(L.gin_bn_ws_bytes(C), torch.uint8, y.device)
    _lib.check(L.gin_bn_stats(y.data_ptr() + 4 * col0, ld, rows, C, bn.weight.data_ptr(), bn.bias.data_ptr(), float(bn.eps), float(bn.momentum),
                              bn.running_mean.data_ptr(), bn.running_var.data_ptr(), bn.num_batches_tracked.data_ptr(), stat.data_ptr(), ws.data_ptr(),
                              _stream()), 'gin_bn_stats')
    return stat


_DUAL = bool(L.gin_forward_operand_is_fp16())        # forward operands fp16: every activation copy also exists in bf16 for wgrad


def _bn_act(y1, col1, ld1, stat1, y2, col2, ld2, stat2, B, level, C, want_b=True, want_f=False, want_w=True):
    """Returns (out_b: the next conv's forward operand copy, out_f: fp32 map, out_w: its bf16 twin = wgrad operand and ReLU mask;
    out_w is out_b itself when the forward format is bf16).  16-bit copies are allocated as torch.bfloat16 containers."""
    dev = y1.device
    out_b = _empty(((B * _P(level) + 2 * B), C), torch.bfloat16, dev) if want_b else None
    out_f = _empty((B * _P(level), C), torch.float32, dev) if want_f else None
    out_w = _empty(((B * _P(level) + 2 * B), C), torch.bfloat16, dev) if (want_w and (_DUAL or not want_b)) else None
    assert y2 is None or y2.dtype == y1.dtype
    _lib.check(L.gin_bn_act_fwd(y1.data_ptr() + y1.element_size() * col1, ld1, stat1.data_ptr(),
                                (y2.data_ptr() + y2.element_size() * col2) if y2 is not None else None, ld2, stat2.data_ptr() if stat2 is not None else None,
                                1 if y1.dtype == torch.float16 else 0, 1,
                                out_b.data_ptr() if want_b else None, out_f.data_ptr() if want_f else None,
                                out_w.data_ptr() if out_w is not None else None, B, level, C, _stream()), 'gin_bn_act_fwd')
    if want_w and out_w is None:
        out_w = out_b
    return out_b, out_f, out_w


def _bn_bwd(dout, mask_b, y, col0, ld, stat, B, level, C, dy_b=None, dy_b_col=0, ldo=0, want_f=False, mask_from_y=True, sync=None):
    """Returns (bstat [4C]: dbeta, dgamma, ..., dy_f or None); writes the bf16 gradient copy into dy_b[:, dy_b_col:dy_b_col+C].
    mask_b must be the activation copy _bn_act produced from (y, stat) with ReLU.  With mask_from_y the kernel re-evaluates the
    mask from y and the BatchNorm constants instead of reading it (include/geniconet_b200.h: relu_from_y): 2 B / element less in
    each pass, step 3.40 -> 3.27 ms on the same box (profiles/r02_ab_mask_*.json).  sync: see _walk; dbeta, dgamma are then this
    rank's sums, the means are over every rank."""
    dev = dout.device
    bstat = _empty(4 * C, torch.float32, dev)
    ws = _empty(L.gin_bn_ws_bytes(C), torch.uint8, dev)
    dy_f = _empty((B * _P(level), C), torch.float32, dev) if want_f else None
    mask, yp, yf16 = mask_b.data_ptr() if mask_b is not None else None, y.data_ptr() + y.element_size() * col0, 1 if y.dtype == torch.float16 else 0
    dyb = (dy_b.data_ptr() + 2 * dy_b_col) if dy_b is not None else None
    if sync is not None:
        rec = _empty(L.gin_bn_sync_record_bytes(C, 0) // 8, torch.float64, dev)
        _lib.check(L.gin_bn_sync_bwd_reduce(dout.data_ptr(), C, mask, yp, ld, yf16, stat.data_ptr(), rec.data_ptr(), ws.data_ptr(), B, level, C,
                                            int(mask_from_y), _stream()), 'gin_bn_sync_bwd_reduce')
        recs = _exchange(rec, sync)
        _lib.check(L.gin_bn_sync_bwd_final(recs.data_ptr(), sync[1], sync[2], C, bstat.data_ptr(), None, _stream()), 'gin_bn_sync_bwd_final')
        _lib.check(L.gin_bn_bwd_apply(dout.data_ptr(), C, mask, yp, ld, yf16, stat.data_ptr(), bstat.data_ptr(), dyb, ldo,
                                      dy_f.data_ptr() if want_f else None, C, B, level, C, int(mask_from_y), _stream()), 'gin_bn_bwd_apply')
        return bstat, dy_f
    _lib.check(L.gin_bn_act_bwd(dout.data_ptr(), C, mask_b.data_ptr() if mask_b is not None else None, y.data_ptr() + y.element_size() * col0, ld,
                                1 if y.dtype == torch.float16 else 0, stat.data_ptr(), bstat.data_ptr(), (dy_b.data_ptr() + 2 * dy_b_col) if dy_b is not None else None, ldo,
                                dy_f.data_ptr() if want_f else None, C, ws.data_ptr(), B, level, C,
                                int(mask_from_y), _stream()), 'gin_bn_act_bwd')
    return bstat, dy_f


def _stem_conv(x, conv):
    """The xyz convolution of a chain's stem (fp32, warp-level kernels).  Returns (plan, packed weights, xs, strides, y, parts):
    y is fp16 with the epilogue's BatchNorm partial sums `parts` = (buffer, rows), or fp32 with parts None."""
    import ctypes
    dev, B = x.device, x.shape[0]
    level, C = conv.subdivisions, conv.out_features
    plan = get_plan(_lib.PLAN_HEXCONV, level, 1, conv.corner_mode, dev)
    packed = _pack(conv.weight.detach().contiguous(), 3, C)
    xs, sb, sp, sc = pixel_strides(x)
    y = _empty((B * _P(level), C), torch.float16 if _Y16 else torch.float32, dev)
    sparts = _empty(L.gin_hexconv_narrow_stats_ws_bytes(C) // 4, torch.float32, dev)
    npart = ctypes.c_int(0)
    rc = L.gin_hexconv_fwd_narrow_stats(plan.host_ptr, plan.dev_ptr, xs.data_ptr(), sb, sp, sc, packed.data_ptr(), conv.bias.data_ptr(),
                                        y.data_ptr(), 1 if _Y16 else 0, B, 3, C, sparts.data_ptr(), ctypes.addressof(npart), _stream())
    if rc == 0 and npart.value > 0:          # output statistics came out of the conv epilogue
        return plan, packed, xs, (sb, sp, sc), y, (sparts, npart.value)
    if rc != 0 and rc != _lib.ERR_UNSUPPORTED:
        _lib.check(rc, 'gin_hexconv_fwd_narrow_stats')
    y = _empty((B * _P(level), C), torch.float32, dev)
    _lib.check(L.gin_hexconv_fwd(plan.host_ptr, plan.dev_ptr, xs.data_ptr(), sb, sp, sc, packed.data_ptr(), conv.bias.data_ptr(),
                                 y.data_ptr(), B, 3, C, _lib.IMPL_AUTO, _stream()), 'gin_hexconv_fwd')
    return plan, packed, xs, (sb, sp, sc), y, None


def _block_stats(ycat, pcat, blk, rows, cout, sync=None):
    """Batch statistics of icobn00 / icobn10 (running statistics updated) from the sibling GEMM's output [rows][conv00 | conv10]."""
    dev = ycat.device
    if sync is not None:
        stat00, stat10 = _empty(4 * cout, torch.float32, dev), _empty(4 * cout, torch.float32, dev)
        _sync_stats(ycat, (0, cout), 2 * cout, rows, cout, pcat, sync, [(blk.icobn00, stat00), (blk.icobn10, stat10)])
    elif pcat is not None:                 # both sibling BatchNorms from the same epilogue sums: one launch
        stat00, stat10 = _empty(4 * cout, torch.float32, dev), _empty(4 * cout, torch.float32, dev)
        bA, bB = blk.icobn00, blk.icobn10
        _lib.check(L.gin_bn_stats_from_parts2(pcat[0].data_ptr(), pcat[1], 2 * cout, rows, cout,
                                              0, bA.weight.data_ptr(), bA.bias.data_ptr(), float(bA.eps), float(bA.momentum), bA.running_mean.data_ptr(),
                                              bA.running_var.data_ptr(), bA.num_batches_tracked.data_ptr(), stat00.data_ptr(),
                                              cout, bB.weight.data_ptr(), bB.bias.data_ptr(), float(bB.eps), float(bB.momentum), bB.running_mean.data_ptr(),
                                              bB.running_var.data_ptr(), bB.num_batches_tracked.data_ptr(), stat10.data_ptr(), _stream()),
                   'gin_bn_stats_from_parts2')
    else:
        stat00 = _bn_stats(ycat, 0, 2 * cout, rows, cout, blk.icobn00, pcat)
        stat10 = _bn_stats(ycat, cout, 2 * cout, rows, cout, blk.icobn10, pcat)
    return stat00, stat10


def _nchw(rows, B, level, C):
    """[B, C, H, W] view, with channels-last strides, of a row-major map [B * P(level)][C]."""
    n = 2 ** level
    return rows.view(B, 5 * n, 2 * n, C).permute(0, 3, 1, 2)


def _rows(t):
    """fp32 [B * P][C] rows of a [B, C, H, W] map; no copy when it has channels-last strides."""
    d = as_channels_last(t).permute(0, 2, 3, 1).reshape(-1, t.shape[1])
    return d if d.is_contiguous() else d.contiguous()


def _cat(blk):
    """The weights of a block's sibling GEMM conv00 | conv10: their wgrad reads the block's input."""
    return (blk.conv00.weight, blk.conv10.weight)


# ------------------------------------------------------------------------------------------------ the chain
def _block(blk, plan_a, plan_b, a_b, pk_cat, pk01, B, lvl, consts, want_h_w, want_b, want_f, want_w, sync=None):
    """A residual block from the forward operand copy a_b of its input: the sibling GEMM conv00 | conv10, BatchNorm 00 / 10,
    relu(bn00) as conv01's operand, conv01, BatchNorm 01, relu(bn01 + bn10).  Batch statistics (running statistics updated) when
    consts is None, else the eval constants consts[bn].  Returns (out_b, out_f, what a backward needs: fp32 / fp16 conv outputs,
    BatchNorm constants and the bf16 twins h_w of conv01's operand and out_w of the output, None where not wanted).  sync: see
    _walk."""
    cin, cout, rows = blk.conv00.in_features, blk.conv00.out_features, B * _P(lvl)
    ycat, pcat = _conv_fwd(plan_a, a_b, pk_cat, blk.conv00.bias.detach(), B, cin, 2 * cout, _P(lvl), bias1=blk.conv10.bias.detach())   # [rows][conv00 | conv10]
    if consts is None:
        stat00, stat10 = _block_stats(ycat, pcat, blk, rows, cout, sync)
    else:
        stat00, stat10 = consts[blk.icobn00][2], consts[blk.icobn10][2]
    h_b, _, h_w = _bn_act(ycat, 0, 2 * cout, stat00, None, 0, 0, None, B, lvl, cout, want_w=want_h_w)
    y01, p01 = _conv_fwd(plan_b, h_b, pk01, blk.conv01.bias.detach(), B, cout, cout, _P(lvl))
    stat01 = _bn_stats(y01, 0, cout, rows, cout, blk.icobn01, p01, sync) if consts is None else consts[blk.icobn01][2]
    out_b, out_f, out_w = _bn_act(y01, 0, cout, stat01, ycat, cout, 2 * cout, stat10, B, lvl, cout, want_b=want_b, want_f=want_f, want_w=want_w)
    return out_b, out_f, dict(ycat=ycat, y01=y01, h_w=h_w, out_w=out_w, stat00=stat00, stat01=stat01, stat10=stat10)


def _block_affine(blk, plan_a, plan_b, a_b, pk_cat, pk01, B, lvl, consts, want_b, want_f):
    """The block in eval mode with each BatchNorm in the epilogue of the convolution that feeds it: relu(bn00(conv00)) as conv01's
    operand, bn10(conv10) as the skip map, then relu(bn01(conv01) + skip).  (out_b, out_f), or None where the epilogue is
    unsupported."""
    cin, cout = blk.conv00.in_features, blk.conv00.out_features
    (sc00, sh00, _), (sc01, sh01, _) = consts[blk.icobn00], consts[blk.icobn01]
    r = _conv_affine(plan_a, a_b, pk_cat, B, cin, 2 * cout, lvl, _span(sc00, 2 * cout), _span(sh00, 2 * cout), cout, cout, (True, False), (False, True))
    if r is not None:
        r = _conv_affine(plan_b, r[0], pk01, B, cout, cout, lvl, sc01, sh01, 0, cout, (want_b, want_f), res=r[3])
    return (r[0], r[1]) if r is not None else None


def _walk(x, mods, consts, twin, copy, record, sync=None):
    """The forward of the chain `mods` (see chain_supported) on x, for the training, forward-only and frozen chains.

    consts: None for batch statistics that update the running statistics, else the eval constants of eval_pairs(mods) in that
    order (with record False the blocks then try the affine epilogue first).  twin(weights): whether to make the bf16 twin of an
    activation copy whose wgrad readers are `weights` (none for a block output that no Down block reads).  copy(nxt): whether to
    make the forward operand copy of the activation that the module nxt reads (None: the chain's output).  record: keep, per
    stage, what a backward needs.  sync: with consts None, sync_group(mods), whose ranks then share the batch statistics.  Returns (fp32 output map [B, C, H, W] with channels-last strides, its forward operand copy or
    None, the stages)."""
    dev, B = x.device, x.shape[0]
    if consts is not None:
        consts = {bn: c for (bn, _), c in zip(eval_pairs(mods), consts)}
    stages = []
    if isinstance(mods[0], IcoConvS2S):                                  # ---- stem: xyz conv (fp32, warp-level kernels) + BN + ReLU
        conv, bn = mods[0], mods[1]
        level, C = conv.subdivisions, conv.out_features
        plan, packed, xs, strides, y, parts = _stem_conv(x, conv)
        stat = _bn_stats(y, 0, C, B * _P(level), C, bn, parts, sync) if consts is None else consts[bn][2]
        act_b, _, act_w = _bn_act(y, 0, C, stat, None, 0, 0, None, B, level, C, want_b=copy(mods[3]), want_w=twin(_cat(mods[3])))
        if record:
            stages.append(dict(kind='stem', plan=plan, xs=xs, strides=strides, y=y, stat=stat, out_w=act_w, C=C, level=level, packed=packed, k=0))
        act_f, i, k = None, 3, 4
    else:                                                                # ---- chain starts on an fp32 map
        blk = mods[0]
        level, C = blk.conv00.subdivisions - (0 if blk._down else 1), blk.conv00.in_features
        xl = as_channels_last(x)
        act_f, act_b, act_w = xl.permute(0, 2, 3, 1).reshape(-1, C), None, None
        if copy(blk):
            plan = get_plan(_lib.PLAN_HEXCONV, level, 1, blk.conv00.corner_mode, dev)
            act_b = cast_bf16(xl, plan, 0, level)
            if twin(_cat(blk)):
                act_w = cast_bf16(xl, plan, 2, level) if _DUAL else act_b
        if record:
            stages.append(dict(kind='input', level=level, C=C, k=0))
        i, k = 0, 0
    # every weight of the chain's tensor-core convolutions is packed by ONE launch
    jobs = []
    for blk in mods[i:]:
        jobs.append((blk.conv00.weight.detach().contiguous(), blk.conv10.weight.detach().contiguous(), blk.conv00.in_features))
        jobs.append((blk.conv01.weight.detach().contiguous(), None, blk.conv01.in_features))
    packs = _pack_many(jobs)
    for j in range(i, len(mods)):
        blk = mods[j]
        nxt = mods[j + 1] if j + 1 < len(mods) else None
        cm = blk.conv00.corner_mode
        cin, cout = blk.conv00.in_features, blk.conv00.out_features
        st = dict(kind='down' if blk._down else 'up', cin=cin, cout=cout, in_level=level, blk=blk, k=k)
        if blk._down:
            lvl = level - 1
            plan_a = get_plan(_lib.PLAN_HEXCONV, level, 2, cm, dev)
            a_b, a_w = act_b, act_w
        else:
            lvl = level + 1
            up_plan = st['up_plan'] = get_plan(_lib.PLAN_UPSAMPLE, level, 1, blk.upsample00.corner_mode, dev)
            plan_a = get_plan(_lib.PLAN_HEXCONV, lvl, 1, cm, dev)
            # upsample straight into the operand copy of the fine level, from the fp32 coarse map (one rounding)
            a_b = _empty((B * _P(lvl) + 2 * B, cin), torch.bfloat16, dev)
            a_w = None
            if twin(_cat(blk)):
                a_w = _empty((B * _P(lvl) + 2 * B, cin), torch.bfloat16, dev) if _DUAL else a_b
            _lib.check(L.gin_upsample_bf16(up_plan.host_ptr, up_plan.dev_ptr, act_f.data_ptr(), 1, a_b.data_ptr(),
                                           a_w.data_ptr() if (_DUAL and a_w is not None) else None, B, cin, _stream()), 'gin_upsample_bf16')
        plan_b = get_plan(_lib.PLAN_HEXCONV, lvl, 1, cm, dev)
        pk_cat, pk01 = packs[2 * (j - i)], packs[2 * (j - i) + 1]
        want_b = copy(nxt)
        want_f = nxt is None or not nxt._down          # an Up block upsamples from the fp32 map (one rounding instead of two)
        r = _block_affine(blk, plan_a, plan_b, a_b, pk_cat, pk01, B, lvl, consts, want_b, want_f) if consts is not None and not record else None
        if r is None:
            out_b, out_f, saved = _block(blk, plan_a, plan_b, a_b, pk_cat, pk01, B, lvl, consts, twin((blk.conv01.weight,)), want_b, want_f,
                                         twin(_cat(nxt) if nxt is not None and nxt._down else ()), sync)
            act_w = saved['out_w']
        else:
            (out_b, out_f), act_w = r, None
        if record:
            # the bf16 twins are kept (wgrad operands, ReLU masks); the forward-format copies die with the forward pass
            st.update(saved, plan_a=plan_a, plan_b=plan_b, a_w=a_w, pk_cat=pk_cat, pk01=pk01, level=lvl)
            stages.append(st)
        act_b, act_f, level, C, k = out_b, out_f, lvl, cout, k + 12
    return _nchw(act_f, B, level, C), act_b, stages


def _block_input_grad(st, dycat_b, B):
    """fp32 gradient of a block's input from the bf16 gradient copy of its sibling GEMM's output: ONE dgrad of conv00 | conv10
    (concatenated along K, which adds the two input gradients), then the upsample's backward for an Up block."""
    cin, cout, lvl = st['cin'], st['cout'], st['level']
    d = _conv_dgrad(st['plan_a'], dycat_b, st['pk_cat'], B, cin, 2 * cout, _P(lvl + 1) if st['kind'] == 'down' else _P(lvl))
    if st['kind'] == 'up':
        upp = st['up_plan']
        d_prev = _empty((B * _P(st['in_level']), cin), torch.float32, d.device)
        _lib.check(L.gin_upsample_bwd(upp.host_ptr, upp.dev_ptr, d.data_ptr(), d_prev.data_ptr(), B, cin, _stream()), 'gin_upsample_bwd')
        d = d_prev
    return d


def _stem_bwd(st, dy_f, B, want_dW, want_db, want_dx):
    """From the fp32 gradient dy_f of the stem convolution's output: (weight gradient, conv-bias gradient, gradient of the xyz
    input), each None where not wanted.  The bias gradient comes out of the weight-gradient kernel."""
    plan, (sb, sp, sc), C, lvl, dev = st['plan'], st['strides'], st['C'], st['level'], dy_f.device
    dW = db = dx = None
    if want_dW:
        dW = _empty((C, 3, 7), torch.float32, dev)
        db = _empty((C,), torch.float32, dev) if want_db else None
        ws = _empty(L.gin_hexconv_wgrad_ws_bytes(3, C), torch.uint8, dev)
        _lib.check(L.gin_hexconv_wgrad(plan.host_ptr, plan.dev_ptr, st['xs'].data_ptr(), sb, sp, sc, dy_f.data_ptr(), dW.data_ptr(),
                                       db.data_ptr() if db is not None else None, ws.data_ptr(), B, 3, C, _lib.IMPL_AUTO, _stream()), 'gin_hexconv_wgrad')
    if want_dx:                     # exact fp32 gather-GEMM: 3 output channels
        dxs = _empty((B * _P(lvl), 3), torch.float32, dev)
        _lib.check(L.gin_hexconv_dgrad(plan.host_ptr, plan.dev_ptr, dy_f.data_ptr(), st['packed'].data_ptr(), dxs.data_ptr(), B, 3, C,
                                       _lib.IMPL_SIMT, _stream()), 'gin_hexconv_dgrad')
        dx = _nchw(dxs, B, lvl, 3)
    return dW, db, dx


class _Chain(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, mods, *params):
        # every twin (the block outputs' are the ReLU masks of backward); the forward copy of every activation but the output, which
        # with bf16 forward operands is its own twin
        ctx.sync = sync_group(mods)
        out, _, ctx.stages = _walk(x, mods, None, lambda ws: True, lambda nxt: nxt is not None or not _DUAL, True, ctx.sync)
        ctx.mods, ctx.B, ctx.x_needs_grad = mods, x.shape[0], x.requires_grad
        return out

    @staticmethod
    def backward(ctx, d_out):
        B, d, dx, sync = ctx.B, _rows(d_out), None, ctx.sync
        plist = chain_params(ctx.mods)          # the Parameter objects, in the order of the gradients this function returns
        grads = [None] * len(plist)
        zmax = max([st['cout'] for st in ctx.stages if st['kind'] in ('down', 'up')] + [1])
        zeros = torch.zeros(zmax, dtype=torch.float32, device=d.device)     # the (exactly zero) gradients of conv biases that feed a BatchNorm
        for st in reversed(ctx.stages):
            k = st['k']
            if st['kind'] in ('down', 'up'):
                cin, cout, lvl, blk = st['cin'], st['cout'], st['level'], st['blk']
                dev = d.device
                dycat_b = _empty((B * _P(lvl) + 2 * B, 2 * cout), torch.bfloat16, dev)
                dy01_b = _empty((B * _P(lvl) + 2 * B, cout), torch.bfloat16, dev)
                # bn01 and bn10 see the same g = d * (out > 0): one pass pair for both
                bs01 = _empty(4 * cout, torch.float32, dev)
                bs10 = _empty(4 * cout, torch.float32, dev)
                ws = _empty(L.gin_bn_pair_ws_bytes(cout), torch.uint8, dev)
                ycat = st['ycat']
                assert st['y01'].dtype == ycat.dtype
                yA, statA, yB, statB = st['y01'].data_ptr(), st['stat01'].data_ptr(), ycat.data_ptr() + ycat.element_size() * cout, st['stat10'].data_ptr()
                yf16 = 1 if ycat.dtype == torch.float16 else 0
                if sync is None:
                    _lib.check(L.gin_bn_act_bwd_pair(d.data_ptr(), cout, st['out_w'].data_ptr(), yA, cout, statA, bs01.data_ptr(), dy01_b.data_ptr(), cout,
                                                     yB, 2 * cout, statB, bs10.data_ptr(), dycat_b.data_ptr() + 2 * cout, 2 * cout, yf16, ws.data_ptr(), B, lvl,
                                                     cout, 1, _stream()), 'gin_bn_act_bwd_pair')
                else:
                    rec = _empty(L.gin_bn_sync_record_bytes(cout, 1) // 8, torch.float64, dev)
                    _lib.check(L.gin_bn_sync_bwd_reduce_pair(d.data_ptr(), cout, st['out_w'].data_ptr(), yA, cout, statA, yB, 2 * cout, statB, yf16,
                                                             rec.data_ptr(), ws.data_ptr(), B, lvl, cout, 1, _stream()), 'gin_bn_sync_bwd_reduce_pair')
                    recs = _exchange(rec, sync)
                    _lib.check(L.gin_bn_sync_bwd_final(recs.data_ptr(), sync[1], sync[2], cout, bs01.data_ptr(), bs10.data_ptr(), _stream()),
                               'gin_bn_sync_bwd_final')
                    _lib.check(L.gin_bn_bwd_apply_pair(d.data_ptr(), cout, st['out_w'].data_ptr(), yA, cout, statA, bs01.data_ptr(), dy01_b.data_ptr(), cout,
                                                       yB, 2 * cout, statB, bs10.data_ptr(), dycat_b.data_ptr() + 2 * cout, 2 * cout, yf16, B, lvl, cout, 1,
                                                       _stream()), 'gin_bn_bwd_apply_pair')
                dW01 = _conv_wgrad(st['plan_b'], st['h_w'], dy01_b, B, cout, cout, out=_dest((blk.conv01.weight,), (cout, cout, 7)))
                d_h = _conv_dgrad(st['plan_b'], dy01_b, st['pk01'], B, cout, cout, _P(lvl))
                bs00, _ = _bn_bwd(d_h, st['h_w'], ycat, 0, 2 * cout, st['stat00'], B, lvl, cout, dycat_b, 0, 2 * cout, sync=sync)
                dWcat = _conv_wgrad(st['plan_a'], st['a_w'], dycat_b, B, cin, 2 * cout, out=_dest(_cat(blk), (2 * cout, cin, 7)))
                d = _block_input_grad(st, dycat_b, B)
                zero_b = zeros[:cout]
                # parameter order of chain_params: conv00 (w, b, gamma, beta) at k, conv01 at k + 4, conv10 at k + 8
                grads[k:k + 12] = [dWcat[:cout], zero_b, bs00[cout:2 * cout], bs00[:cout], dW01, zero_b, bs01[cout:2 * cout], bs01[:cout],
                                   dWcat[cout:], zero_b, bs10[cout:2 * cout], bs10[:cout]]
                n = 12
            elif st['kind'] == 'stem':
                C = st['C']
                bs, dy_f = _bn_bwd(d, st['out_w'], st['y'], 0, C, st['stat'], B, st['level'], C, want_f=True, sync=sync)
                dW, db, dx = _stem_bwd(st, dy_f, B, True, True, ctx.x_needs_grad)
                grads[0:4] = [dW, db, bs[C:2 * C], bs[:C]]
                n = 4
            else:   # 'input': gradient of the fp32 map the chain started from
                dx, n = _nchw(d, B, st['level'], st['C']), 0
            if _grad_sink is not None and n:
                _grad_sink([(plist[q], grads[q]) for q in reversed(range(k, k + n))])     # last parameter first
        return (dx, None) + tuple(grads)


def run_chain(x, mods):
    """Forward of the module list `mods` (see chain_supported) on the fused path; x fp32 CUDA, returns the fp32 output map."""
    mods = list(mods)
    return _Chain.apply(x, mods, *chain_params(mods))


# ------------------------------------------------------------------------------------------------ forward-only chain (inference)
_EVAL_CACHE = {}


def _bn_table(pairs):
    """Device table of GinBnEvalEntry (include/geniconet_b200.h) for `pairs` = [(BatchNorm2d, conv bias or None)] and the fp32
    buffer it fills: per entry scale [C], shift [C] (conv bias folded in), stat [4][C] (gin_bn_act_fwd layout, no bias).  Cached
    per set of parameter storages: the table holds pointers only, so in-place load_state_dict needs no rebuild, and a captured
    graph reads the current values at every replay."""
    # num_features too: a BatchNorm created after another one died can get its id() and, from the caching allocator, the same
    # storage addresses with a different width
    key = tuple((id(bn), bn.num_features, bn.weight.data_ptr(), bn.bias.data_ptr(), bn.running_mean.data_ptr(), bn.running_var.data_ptr(),
                 float(bn.eps), b.data_ptr() if b is not None else 0) for bn, b in pairs)
    hit = _EVAL_CACHE.get(key)
    if hit is not None:
        return hit
    import ctypes
    import numpy as np
    dev = pairs[0][0].weight.device
    sizes = [bn.num_features for bn, _ in pairs]
    S = sum(sizes)
    buf = torch.empty(6 * S, dtype=torch.float32, device=dev)      # [all scales | all shifts | all stats]: consecutive entries adjacent
    rec = np.dtype([('p', np.uint64, 8), ('eps', np.float32), ('C', np.int32)])
    assert rec.itemsize == 72
    tab = np.zeros(len(pairs), dtype=rec)
    views, off = [], 0
    for k, ((bn, b), C) in enumerate(zip(pairs, sizes)):
        sc, sh, st = buf[off:off + C], buf[S + off:S + off + C], buf[2 * S + 4 * off:2 * S + 4 * (off + C)]
        off += C
        tab[k]['p'] = [bn.weight.data_ptr(), bn.bias.data_ptr(), bn.running_mean.data_ptr(), bn.running_var.data_ptr(),
                       b.data_ptr() if b is not None else 0, sc.data_ptr(), sh.data_ptr(), st.data_ptr()]
        tab[k]['eps'], tab[k]['C'] = bn.eps, C
        views.append((sc, sh, st))
    table = torch.from_numpy(tab.view(np.uint8).copy()).to(dev)
    hit = _EVAL_CACHE[key] = (table, len(pairs), max(sizes), buf, views)
    return hit


def _eval_consts(pairs):
    """[(scale, shift, stat)] per pair, computed on the device from the current parameters and running statistics (one launch)."""
    table, n, cmax, _, views = _bn_table(pairs)
    _lib.check(L.gin_bn_eval_consts(table.data_ptr(), n, cmax, _stream()), 'gin_bn_eval_consts')
    return views


def _span(t, n):
    """n elements of t's storage from t's first element on: the constants of consecutive table entries as one vector"""
    return t.as_strided((n,), (1,))


def _conv_affine(plan, xb, packed, B, cin, cout, level, scale, shift, relu_split, split, want0, want1=(False, False), res=None):
    """Convolution with eval-mode BatchNorm in the epilogue (gin_hexconv_fwd_affine).  want0 / want1 = (operand copy, fp32 map) of
    the columns < split / >= split.  Returns [out0_b, out0_f, out1_b, out1_f] (None where not wanted), or None when the epilogue
    does not support this plan and size."""
    dev, rows = xb.device, B * _P(level)
    outs = []
    for (wb, wf), width in ((want0, split), (want1, cout - split)):
        outs.append(_empty((rows + 2 * B, width), torch.bfloat16, dev) if wb else None)
        outs.append(_empty((rows, width), torch.float32, dev) if wf else None)
    ring = _empty(L.gin_hexconv_affine_ring_bytes(B, cout) // 4, torch.float32, dev) if (want0[0] or want1[0]) else None
    ptr = lambda t: t.data_ptr() if t is not None else None
    rc = L.gin_hexconv_fwd_affine(plan.host_ptr, plan.dev_ptr, xb.data_ptr(), packed.data_ptr(), scale.data_ptr(), shift.data_ptr(), relu_split,
                                  ptr(res), res.shape[1] if res is not None else 0, 1 if res is not None and res.dtype == torch.float16 else 0,
                                  split, *[ptr(t) for t in outs], ptr(ring), B, cin, cout, _stream())
    if rc == _lib.ERR_UNSUPPORTED:
        return None
    _lib.check(rc, 'gin_hexconv_fwd_affine')
    return outs


def eval_pairs(mods):
    """(BatchNorm, conv bias or None) of every BatchNorm of a chain, in the order infer_chain reads their constants; the stem's
    BatchNorm is applied by gin_bn_act_fwd to a map that already holds the conv bias."""
    pairs = []
    for m in mods:
        if isinstance(m, _BN):
            pairs.append((m, None))
        elif _is_block(m):
            pairs += [(m.icobn00, m.conv00.bias), (m.icobn10, m.conv10.bias), (m.icobn01, m.conv01.bias)]
    return pairs


def infer_chain(x, mods, want_operand=False):
    """Forward-only execution of the chain `mods` (see chain_supported): no autograd, nothing saved, no bf16 wgrad twins.

    Eval mode (every BatchNorm has training == False): the BatchNorms use their running statistics; the constants of all of them
    come from one launch (gin_bn_eval_consts) and are applied in the epilogue of the convolution that feeds them
    (gin_hexconv_fwd_affine), with gin_hexconv_fwd_bf16_stats2 + gin_bn_act_fwd wherever that epilogue is unsupported and for the
    stem.  Train mode (under no_grad): the training chain's forward kernels with batch statistics; output and running statistics are
    bit for bit those of _Chain.forward.

    Returns (fp32 output map [B, C, H, W] with channels-last strides, its 16-bit forward operand copy when want_operand else None)."""
    mods = list(mods)
    consts = None if mods[-1].icobn01.training else _eval_consts(eval_pairs(mods))
    out, act_b, _ = _walk(x, mods, consts, lambda ws: False, lambda nxt: nxt is not None or want_operand, False)
    return out, act_b


# ------------------------------------------------------------------------------------------------ frozen BatchNorm (eval mode with grad)
def frozen_supported(mods):
    """chain_supported, and every BatchNorm at most 256 wide (gin_bn_eval_bwd keeps its constants in shared memory)."""
    return chain_supported(mods) and all(bn.num_features <= 256 for bn, _ in eval_pairs(mods))


def _own_consts(pairs):
    """The eval constants of `pairs` (see _eval_consts) in a buffer of this call's own: _bn_table's buffer is shared by every call
    on the same parameters and rewritten by each, while a backward must see the constants of its own forward."""
    _, _, _, buf, views = _bn_table(pairs)
    _eval_consts(pairs)
    own = buf.clone()
    return [tuple(own[v.storage_offset():v.storage_offset() + v.numel()] for v in vs) for vs in views]


def _eval_bwd(dout, y, col0, ld, stat, B, level, C, bsum, dy_b=None, dy_b_col=0, ldo=0, want_f=False):
    """gin_bn_eval_bwd with the ReLU mask re-evaluated from y.  Returns dy_f (or None); writes bsum [3C] when given and the bf16
    gradient copy into dy_b[:, dy_b_col:dy_b_col+C]."""
    dev = dout.device
    dy_f = _empty((B * _P(level), C), torch.float32, dev) if want_f else None
    ws = _empty(L.gin_bn_eval_bwd_ws_bytes(C), torch.uint8, dev) if bsum is not None else None
    ptr = lambda t: t.data_ptr() if t is not None else None
    _lib.check(L.gin_bn_eval_bwd(dout.data_ptr(), C, None, y.data_ptr() + y.element_size() * col0, ld, 1 if y.dtype == torch.float16 else 0,
                                 stat.data_ptr(), ptr(bsum), (dy_b.data_ptr() + 2 * dy_b_col) if dy_b is not None else None, ldo, ptr(dy_f), C,
                                 ptr(ws), B, level, C, 1, _stream()), 'gin_bn_eval_bwd')
    return dy_f


def _take_sums(grads, need, k, bs, C):
    """conv bias, gamma, beta (parameters k + 1 .. k + 3 of chain_params) from bsum = [dbeta | dgamma | conv-bias gradient]"""
    for kk, g in ((k + 1, bs[2 * C:]), (k + 2, bs[C:2 * C]), (k + 3, bs[:C])):
        grads[kk] = g if need[kk] else None


class _FrozenChain(torch.autograd.Function):
    """The chain with every BatchNorm in eval mode and grad enabled: the training chain's forward kernels with the running-statistic
    constants (nothing is updated), and a backward through gin_bn_eval_bwd(_pair).  Weight gradients are computed only for weights
    that need them; BatchNorm sums only where gamma, beta or the conv bias needs a gradient."""

    @staticmethod
    def forward(ctx, x, mods, *params):
        # twins only for weights that need a gradient, forward copies only where a Down block reads them
        out, _, ctx.stages = _walk(x, mods, _own_consts(eval_pairs(mods)), lambda ws: any(w.requires_grad for w in ws),
                                   lambda nxt: nxt is not None and nxt._down, True)
        ctx.B, ctx.need, ctx.x_needs_grad = x.shape[0], [p.requires_grad for p in params], x.requires_grad
        return out

    @staticmethod
    def backward(ctx, d_out):
        B, stages, need, d, dx = ctx.B, ctx.stages, ctx.need, _rows(d_out), None
        grads = [None] * len(need)
        # upstream[s]: something before stage s (an earlier stage's parameter, or x) needs a gradient
        upstream, acc = [], ctx.x_needs_grad
        for st in stages:
            upstream.append(acc)
            if st['kind'] != 'input':
                acc = acc or any(need[st['k']:st['k'] + (4 if st['kind'] == 'stem' else 12)])
        dev = d.device
        sums = lambda k, C: _empty(3 * C, torch.float32, dev) if any(need[k + 1:k + 4]) else None
        ptr = lambda t: t.data_ptr() if t is not None else None
        for s in range(len(stages) - 1, -1, -1):
            st = stages[s]
            if st['kind'] in ('down', 'up'):
                cin, cout, lvl, k = st['cin'], st['cout'], st['level'], st['k']
                # parameter order of chain_params: conv00 (w, b, gamma, beta) at k, conv01 at k + 4, conv10 at k + 8
                bs00, bs01, bs10 = sums(k, cout), sums(k + 4, cout), sums(k + 8, cout)
                dycat_b = _empty((B * _P(lvl) + 2 * B, 2 * cout), torch.bfloat16, dev)
                dy01_b = _empty((B * _P(lvl) + 2 * B, cout), torch.bfloat16, dev)
                ws = _empty(L.gin_bn_eval_bwd_ws_bytes(cout), torch.uint8, dev) if (bs01 is not None or bs10 is not None) else None
                ycat = st['ycat']
                _lib.check(L.gin_bn_eval_bwd_pair(d.data_ptr(), cout, None, st['y01'].data_ptr(), cout, st['stat01'].data_ptr(), ptr(bs01),
                                                  dy01_b.data_ptr(), cout, ycat.data_ptr() + ycat.element_size() * cout, 2 * cout,
                                                  st['stat10'].data_ptr(), ptr(bs10), dycat_b.data_ptr() + 2 * cout, 2 * cout,
                                                  1 if ycat.dtype == torch.float16 else 0, ptr(ws), B, lvl, cout, 1, _stream()), 'gin_bn_eval_bwd_pair')
                if need[k + 4]:
                    grads[k + 4] = _conv_wgrad(st['plan_b'], st['h_w'], dy01_b, B, cout, cout)
                d_h = _conv_dgrad(st['plan_b'], dy01_b, st['pk01'], B, cout, cout, _P(lvl))
                _eval_bwd(d_h, ycat, 0, 2 * cout, st['stat00'], B, lvl, cout, bs00, dycat_b, 0, 2 * cout)
                if need[k] or need[k + 8]:
                    dWcat = _conv_wgrad(st['plan_a'], st['a_w'], dycat_b, B, cin, 2 * cout)
                    grads[k], grads[k + 8] = (dWcat[:cout] if need[k] else None), (dWcat[cout:] if need[k + 8] else None)
                for kk, bs in ((k, bs00), (k + 4, bs01), (k + 8, bs10)):
                    if bs is not None:
                        _take_sums(grads, need, kk, bs, cout)
                if not upstream[s]:
                    break
                d = _block_input_grad(st, dycat_b, B)
            elif st['kind'] == 'stem':
                C = st['C']
                bs = sums(0, C)
                if not (need[0] or bs is not None or ctx.x_needs_grad):
                    break
                dy_f = _eval_bwd(d, st['y'], 0, C, st['stat'], B, st['level'], C, bs, want_f=True)
                grads[0], _, dx = _stem_bwd(st, dy_f, B, need[0], False, ctx.x_needs_grad)
                if bs is not None:
                    _take_sums(grads, need, 0, bs, C)
            else:
                dx = _nchw(d, B, st['level'], st['C'])
        return (dx, None) + tuple(grads)


def run_frozen_chain(x, mods):
    """Forward of the module list `mods` (see frozen_supported) with every BatchNorm in eval mode, differentiable: the running
    statistics are used and left untouched, gradients flow to x and to every parameter that requires one."""
    mods = list(mods)
    return _FrozenChain.apply(x, mods, *chain_params(mods))


def latent_supported(mu, logvar):
    """The VAE's mu / logvar heads (IcoConvS2S stride 2 + BatchNorm, models.py _latent_head) in eval mode, without hooks."""
    for head in (mu, logvar):
        mods = list(head)
        if len(mods) != 2 or not isinstance(mods[0], IcoConvS2S) or not isinstance(mods[1], _BN):
            return False
        c, bn = mods
        if (c.stride != 2 or c.bias is None or getattr(c, 'impl', 0) != 0 or bn.training or not bn.affine or not bn.track_running_stats
                or c.in_features % 64 or c.out_features % 64):
            return False
        if any(m._forward_hooks or m._forward_pre_hooks for m in [head] + mods):
            return False
    a, b = mu[0], logvar[0]
    return (a.in_features, a.out_features, a.subdivisions, a.corner_mode) == (b.in_features, b.out_features, b.subdivisions, b.corner_mode)


def infer_latent(h_b, mu, logvar, B):
    """mu and logvar heads as ONE stride-2 GEMM with two fp32 destinations; h_b = the operand copy of their common input.
    Returns (mu, logvar) as [B, C, H, W] maps with channels-last strides, or None when the epilogue does not support the size."""
    c0, c1 = mu[0], logvar[0]
    cin, cout, lvl = c0.in_features, c0.out_features, c0.subdivisions - 1
    (sa, ha, _), _ = _eval_consts([(mu[1], c0.bias), (logvar[1], c1.bias)])
    packed = _pack_many([(c0.weight.detach().contiguous(), c1.weight.detach().contiguous(), cin)])[0]
    plan = get_plan(_lib.PLAN_HEXCONV, c0.subdivisions, 2, c0.corner_mode, h_b.device)
    r = _conv_affine(plan, h_b, packed, B, cin, 2 * cout, lvl, _span(sa, 2 * cout), _span(ha, 2 * cout), 0, cout, (False, True), (False, True))
    if r is None:
        return None
    return _nchw(r[1], B, lvl, cout), _nchw(r[3], B, lvl, cout)


# ------------------------------------------------------------------ decoder head: Conv2d(64, 3, 1) -> Tanh (models.py:151-154)
def head_supported(head, x):
    """head = nn.Sequential(Conv2d 1x1 64->3 with bias, Tanh) without hooks, x a dense fp32 CUDA map."""
    mods = list(head)
    if len(mods) != 2 or not isinstance(mods[0], torch.nn.Conv2d) or not isinstance(mods[1], torch.nn.Tanh):
        return False
    c = mods[0]
    if (c.kernel_size != (1, 1) or c.stride != (1, 1) or c.padding != (0, 0) or c.groups != 1 or c.bias is None
            or c.in_channels != 64 or c.out_channels != 3 or c.weight.dtype != torch.float32):
        return False
    if any(m._forward_hooks or m._forward_pre_hooks or m._backward_hooks for m in [head] + mods):
        return False
    return x.is_cuda and x.dtype == torch.float32 and x.dim() == 4 and x.shape[1] == 64


class _Head(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias):
        B, C, H, W = x.shape
        xs = as_channels_last(x)                              # [B*P][64] in memory; no copy after a fused chain
        w = weight.reshape(3, C).contiguous()
        y = torch.empty((B, 3, H, W), dtype=torch.float32, device=x.device)
        _lib.check(_lib.lib.gin_head_fwd(xs.data_ptr(), w.data_ptr(), bias.data_ptr(), y.data_ptr(), B, H * W, C, 3, _stream()), 'gin_head_fwd')
        ctx.save_for_backward(xs, w, y)
        return y

    @staticmethod
    def backward(ctx, dy):
        xs, w, y = ctx.saved_tensors
        B, C, H, W = xs.shape
        dy = dy.contiguous()
        dx = torch.empty_strided(xs.shape, xs.stride(), dtype=torch.float32, device=xs.device)
        dw = torch.empty((3, C, 1, 1), dtype=torch.float32, device=xs.device)
        db = torch.empty(3, dtype=torch.float32, device=xs.device)
        ws = _empty(_lib.lib.gin_head_ws_bytes(), torch.uint8, xs.device)
        _lib.check(_lib.lib.gin_head_bwd(xs.data_ptr(), w.data_ptr(), y.data_ptr(), dy.data_ptr(), dx.data_ptr(), dw.data_ptr(), db.data_ptr(),
                                         ws.data_ptr(), B, H * W, C, 3, _stream()), 'gin_head_bwd')
        return dx, dw, db


def run_head(head, x):
    return _Head.apply(x, head[0].weight, head[0].bias)
