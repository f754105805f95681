"""Whole-stack autograd for the residual GCN of the botnet path (gcn_model.py:86-106 with
residual_hop=1, ReLU activations, additive node model, aggr='add'):

    x_{n+1} = act_n( relu( A_hat (x_n W_n) + b_n ) + x_n R_n^T + r_n ),   act_n = ReLU, identity for the last layer

One Function for all L layers: the degree factors are applied once per layer by the transform that
produces the messages (x~w = pre * xW), so the aggregation needs no per-edge weight; both ReLU
masks of the backward are folded into operand loads; no autograd graph, no [N,H] temporaries
beyond the saved layer outputs.  Per layer: forward = transform, aggregation, residual transform
(3 launches); backward = weight-gradient x2, transform x2, mask/scale, transposed aggregation.
"""
import os

import torch

from . import ops

FUSED_WIDTHS = (16, 32, 64, 128)
# row-local backward of the hidden-32 stack: tcgen05 / TMEM pipeline (0.64 ms per layer at the botnet batch)
# or the mma.sync kernel (0.81 ms); both pass the same parity tests
BWD_TENSOR_MEMORY = True
# hidden-32 stack: aggregate-then-transform forward on tcgen05 (csrc/gcn_fwd_tc.cu; one [N,32] read + one write per
# layer) or the transform-then-aggregate kernels of round 1 (csrc/gcn_layer.cu); both pass the same parity tests
FORWARD_AGGREGATE_FIRST = True
# aggregate-then-transform stack: transposed aggregation + row-local backward as ONE launch per layer
# (csrc/gcn_bwd_fused.cu: no dxw array, 0.9 GB less DRAM traffic per layer) instead of two.  Same parity tests,
# identical from run to run — but measured SLOWER at the botnet batch (1.45 ms against 0.48 + 0.61 ms: the per-row
# operand-image work needs more warps than fit next to a 16-warp gather), so it is off by default
BWD_FUSED = os.environ.get("MGCN_BWD_FUSED", "0") == "1"


def dropout_seed(device):
    """The seed of one forward's dropout masks: one int64 drawn on the device from torch's CUDA generator, so
    torch.manual_seed / torch.cuda.set_rng_state reproduce it and every replay of a captured CUDA graph draws anew.
    The only source of randomness of the stack (a test pins the masks by replacing this function)."""
    return torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), device=device, dtype=torch.int64)


def _dropout_masks(x, L, W, p):
    """(keep int32 [L, N, W], scale 1 / (1 - p)) for 0 < p < 1, else (None, None): the masks of all L layers in one
    launch (csrc/dropout.cu); dropped with the forward's locals — the backward reads only the saved ReLU masks"""
    if not p:
        return None, None
    keep = ops.dropout_keep_bits_impl(dropout_seed(x.device), L, x.size(0), W, p)
    return keep, 1.0 / (1.0 - p)


def _scaled_post(post, scale, n, like):
    """the per-target factor of the backward with the dropout scale folded in: kept * relu'(h) is in the mask, the scale
    rides on the row vector the backward multiplies by anyway (exact at p = 0.5, one rounding otherwise)"""
    if scale is None:
        return post
    return post * scale if post is not None else torch.full((n,), scale, dtype=torch.float32, device=like.device)


class _ResidualGCNStack(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, graph, pre, post, has_bias, last_relu, p, *params):
        per = 4 if has_bias else 3
        L = len(params) // per
        layers = [params[i * per:(i + 1) * per] for i in range(L)]
        xs, hs = [x.contiguous()], []
        fwd = graph.fwd_plain
        keep, scale = _dropout_masks(x, L, (max(lp[0].size(1) for lp in layers) + 31) // 32, p)
        xw = ops.linear_impl(xs[0], layers[0][0], False, row_scale=pre)
        for n, lp in enumerate(layers):
            w, b = lp[0], (lp[1] if has_bias else None)
            res_w, res_b = lp[-2], lp[-1]
            h = ops.aggregate_prescaled_impl(fwd, xw, post, 0, b, None, 1)
            if keep is not None:
                ops.dropout_apply_impl(h, keep[n], scale)      # saved as dropped: its ReLU mask is h > 0
            relu_out = last_relu or n < L - 1
            xn = ops.linear_impl(xs[n], res_w, True, res_b, h, 1 if relu_out else 0)
            hs.append(h)
            xs.append(xn)
            if n + 1 < L:
                xw = ops.linear_impl(xn, layers[n + 1][0], False, row_scale=pre)
        ctx.graph, ctx.cfg = graph, (L, per, has_bias, last_relu)
        ctx.pre, ctx.post = pre, post
        # dropout scale of the backward: on the node-model output before the bias gradient is taken, else with post
        ctx.unit_scale = None
        if scale is not None and has_bias:
            ctx.unit_scale = torch.full((x.size(0),), scale, dtype=torch.float32, device=x.device)
        elif scale is not None:
            ctx.post = _scaled_post(post, scale, x.size(0), x)
        ctx.save_for_backward(*xs, *hs, *params)
        return xs[-1]

    @staticmethod
    def backward(ctx, g):
        L, per, has_bias, last_relu = ctx.cfg
        saved = ctx.saved_tensors
        xs, hs, params = saved[:L + 1], saved[L + 1:2 * L + 1], saved[2 * L + 1:]
        layers = [params[i * per:(i + 1) * per] for i in range(L)]
        pre, post, bwd = ctx.pre, ctx.post, ctx.graph.bwd_plain
        grads = [None] * len(params)
        g = g.contiguous()
        need_x = ctx.needs_input_grad[0]
        for n in reversed(range(L)):
            lp = layers[n]
            w, res_w = lp[0], lp[-2]
            omask = xs[n + 1] if (last_relu or n < L - 1) else None
            d_res_w, d_res_b = ops.linear_wgrad_impl(xs[n], g, True, True, omask)
            need_dx = n > 0 or need_x
            dxres = ops.linear_impl(g, res_w, False, xmask=omask) if need_dx else None
            if has_bias:
                gsu = ops.masked_scale_impl(g, omask, hs[n], ctx.unit_scale)
                grads[n * per + 1] = gsu.sum(0)
                gs = ops.masked_scale_impl(gsu, None, None, post) if post is not None else gsu
            else:
                gs = ops.masked_scale_impl(g, omask, hs[n], post)
            dxw = ops.aggregate_prescaled_impl(bwd, gs, pre, 0, None, None, 0)
            grads[n * per] = ops.linear_wgrad_impl(xs[n], dxw, False, False)[0]
            grads[n * per + per - 2] = d_res_w
            grads[n * per + per - 1] = d_res_b
            if need_dx:
                g = ops.linear_impl(dxw, w, True, add=dxres)
        return (g if need_x else None, None, None, None, None, None, None, *grads)


class _ResidualGCNStack32(torch.autograd.Function):
    """hidden width 32, no node-model bias: one fused launch per layer forward (aggregation + both
    dense products on the tensor pipe, csrc/gcn_layer.cu), transposed aggregation + one row-local
    launch per layer backward.  Saved per layer: the layer input x_n and one mask word per row."""

    @staticmethod
    def forward(ctx, x, graph, pre, post, last_relu, *params):
        L = len(params) // 3
        layers = [params[i * 3:(i + 1) * 3] for i in range(L)]
        fwd = graph.fwd_plain
        x0 = x.contiguous()
        xs, hmasks = [x0], []
        # A first layer of small input width is aggregated BEFORE its transform — (A_hat x) W instead of
        # A_hat (x W): the gather moves H_in instead of 32 floats per entry, and its backward needs no
        # transposed aggregation at all:  dW_0 = s^T gs_0  with  s = sum_j pre_j x_j  saved here.  The layer's
        # two [N,32] operands (s W_0 and x R_0^T + r_0) are formed inside its launch (mgcn_gcn_first_layer_fwd).
        agg_first = x0.size(1) <= 4 and not ctx.needs_input_grad[0]
        s0 = resid0 = None
        if agg_first:
            xs0 = x0 * pre.unsqueeze(1) if pre is not None else x0            # pre_j x_j, one rounding as in the gather
            s0 = ops.spmm_impl(fwd, xs0)                                      # [N, H_in]
        else:
            resid0 = ops.linear_impl(x0, layers[0][1], True, layers[0][2])    # x0 R0^T + r0
            m = ops.linear_impl(x0, layers[0][0], False, row_scale=pre)       # messages of layer 0
        for n in range(L):
            w_next = layers[n + 1][0] if n + 1 < L else None
            act_out = 1 if (last_relu or n < L - 1) else 0
            if n == 0 and agg_first:
                xn, m, hm = ops.gcn_first_layer_fwd_impl(s0, x0, layers[0][0], layers[0][1], layers[0][2], w_next,
                                                         pre, post, act_out)
            else:
                xn, m, hm = ops.gcn_layer_fwd_impl(
                    fwd, m, xs[n] if n > 0 else None, resid0 if n == 0 else None,
                    layers[n][1], layers[n][2], w_next, None, pre, post, act_out)
            xs.append(xn)
            hmasks.append(hm)
        ctx.agg_first = agg_first
        ctx.s0 = s0
        ctx.graph, ctx.cfg = graph, (L, last_relu)
        ctx.pre, ctx.post = pre, post
        ctx.save_for_backward(*xs, *hmasks, *params)
        return xs[-1]

    @staticmethod
    def backward(ctx, g):
        L, last_relu = ctx.cfg
        saved = ctx.saved_tensors
        xs, hmasks, params = saved[:L + 1], saved[L + 1:2 * L + 1], saved[2 * L + 1:]
        layers = [params[i * 3:(i + 1) * 3] for i in range(L)]
        pre, post, bwd = ctx.pre, ctx.post, ctx.graph.bwd_plain
        grads = [None] * len(params)
        gy = g.contiguous()
        if last_relu:
            gy = ops.relu_backward_impl(gy, xs[L])
        gs = ops.mask_bits_scale_impl(gy, hmasks[L - 1], post)
        for n in range(L - 1, 0, -1):
            dxw = ops.aggregate_prescaled_impl(bwd, gs, pre, 0, None, None, 0)
            gy_prev, gs_prev, dw, drw, drb = ops.gcn_layer_bwd_impl(
                dxw, gy, xs[n], layers[n][0], layers[n][1], hmasks[n - 1], post, True, BWD_TENSOR_MEMORY)
            grads[3 * n], grads[3 * n + 1], grads[3 * n + 2] = dw, drw, drb
            gy, gs = gy_prev, gs_prev
        grads[1], grads[2] = ops.linear_wgrad_impl(xs[0], gy, True, True)
        gx = None
        if ctx.agg_first:
            grads[0] = ops.linear_wgrad_impl(ctx.s0, gs, False, False)[0]    # dW0 = s0^T gs0
        else:
            dxw = ops.aggregate_prescaled_impl(bwd, gs, pre, 0, None, None, 0)
            grads[0] = ops.linear_wgrad_impl(xs[0], dxw, False, False)[0]
            if ctx.needs_input_grad[0]:
                gx = ops.linear_impl(gy, layers[0][1], False)
                gx = ops.linear_impl(dxw, layers[0][0], True, add=gx)
        return (gx, None, None, None, None, *grads)


class _ResidualGCNStack32AT(torch.autograd.Function):
    """hidden width 32, no node-model bias, AGGREGATE-THEN-TRANSFORM: (A_hat x) W instead of A_hat (x W).  One
    tcgen05 launch per layer forward (csrc/gcn_fwd_tc.cu) that reads one [N,32] array and writes one: activations are
    stored as z_n = sigma (.) x_n (sigma = the per-source degree factor, 1 where that factor is 0 — such a row is
    never a source when the degree is the graph's own out-degree), so the gather needs no per-edge weight and no
    separate message array; the row-local terms divide sigma out per row.  Saved per layer: z_n and one mask word
    per row.  Backward: dW_n = x_n^T (A_hat^T ga), dx = (A_hat^T ga) W_n^T + gy R_n — the transposed aggregation of
    the masked gradient, then the row-local tcgen05 launch."""

    @staticmethod
    def forward(ctx, x, graph, pre, post, last_relu, p, *params):
        L = len(params) // 3
        layers = [params[i * 3:(i + 1) * 3] for i in range(L)]
        fwd = graph.fwd_plain
        x0 = x.contiguous()
        sigma = None
        if pre is not None:
            sigma = torch.where(pre > 0, pre, torch.ones_like(pre))
        # dropout: applied in the layer kernels' epilogues, the dropped entries cleared in the ReLU mask words
        keep, scale = _dropout_masks(x0, L, 1, p)
        drop = (lambda n: {"keep": keep[n], "keep_scale": scale}) if keep is not None else (lambda n: {})
        zs, hmasks = [], []
        agg_first = x0.size(1) <= 4
        s0 = None
        if agg_first:
            xs0 = x0 * pre.unsqueeze(1) if pre is not None else x0            # pre_j x_j, one rounding as in the gather
            s0 = ops.spmm_impl(fwd, xs0)                                      # [N, H_in]
            z, _, hm = ops.gcn_first_layer_fwd_impl(
                s0, x0, layers[0][0], layers[0][1], layers[0][2], None, None, post,
                1 if (last_relu or L > 1) else 0, out_scale=sigma if L > 1 else None, **drop(0))
            zs.append(None)
            hmasks.append(hm)
            first = 1
        else:
            z = x0 * sigma.unsqueeze(1) if sigma is not None else x0
            first = 0
        for n in range(first, L):
            zs.append(z)
            z, hm = ops.gcn_layer_fwd_tc_impl(
                fwd, z, layers[n][0], layers[n][1], layers[n][2], None, sigma, post,
                sigma if n < L - 1 else None, 1 if (last_relu or n < L - 1) else 0, **drop(n))
            hmasks.append(hm)
        ctx.agg_first = agg_first
        ctx.graph, ctx.cfg = graph, (L, last_relu)
        # the backward reads `post` only where it scales a gradient by the mask words: the dropout scale goes there
        ctx.save_for_backward(x0, s0, pre, _scaled_post(post, scale, x0.size(0), x0), sigma, z if last_relu else None,
                              *[t for t in zs if t is not None], *hmasks, *params)
        return z

    @staticmethod
    def backward(ctx, g):
        L, last_relu = ctx.cfg
        saved = ctx.saved_tensors
        x0, s0, pre, post, sigma, out = saved[:6]
        nz = L - 1 if ctx.agg_first else L
        zs = list(saved[6:6 + nz])
        if ctx.agg_first:
            zs = [None] + zs
        hmasks = saved[6 + nz:6 + nz + L]
        params = saved[6 + nz + L:]
        layers = [params[i * 3:(i + 1) * 3] for i in range(L)]
        bwd = ctx.graph.bwd_plain
        grads = [None] * len(params)
        gy = g.contiguous()
        if last_relu:
            gy = ops.relu_backward_impl(gy, out)
        gs = ops.mask_bits_scale_impl(gy, hmasks[L - 1], post)
        last = 1 if ctx.agg_first else 0
        for n in range(L - 1, last - 1, -1):
            want_prev = n > 0
            if BWD_FUSED:
                gy_prev, gs_prev, dw, drw, drb = ops.gcn_layer_bwd_fused_impl(
                    bwd, gs, gy, zs[n], layers[n][0], layers[n][1], hmasks[n - 1] if want_prev else None, post,
                    row_scale=pre, x_scale=sigma, want_prev=want_prev)
            else:
                dxw = ops.aggregate_prescaled_impl(bwd, gs, pre, 0, None, None, 0)
                gy_prev, gs_prev, dw, drw, drb = ops.gcn_layer_bwd_impl(
                    dxw, gy, zs[n], layers[n][0], layers[n][1], hmasks[n - 1] if want_prev else None, post,
                    want_prev, True, x_scale=sigma)
            grads[3 * n], grads[3 * n + 1], grads[3 * n + 2] = dw, drw, drb
            if want_prev:
                gy, gs = gy_prev, gs_prev
        if ctx.agg_first:
            grads[1], grads[2] = ops.linear_wgrad_impl(x0, gy, True, True)
            grads[0] = ops.linear_wgrad_impl(s0, gs, False, False)[0]    # dW0 = s0^T gs0
        return (None, None, None, None, None, None, *grads)


def residual_gcn_stack(x, graph, pre, post, layer_params, has_bias, last_relu=False, aggregate_first=True,
                       dropout=0.0):
    """layer_params: per layer (weight_node [Hin,H], [bias [H]], residual.weight [H,Hin],
    residual.bias [H]).  pre/post: per-source / per-target degree factors (either may be None).
    dropout: p of nn.Dropout on every layer's node-model output (0 <= p < 1; pass 0 outside training).
    Returns None where the stack does not take dropout (the round-1 hidden-32 kernels, chosen for an x that requires
    grad or a degree with zeros): the caller then composes the layers one by one."""
    if not 0.0 <= dropout < 1.0:
        raise ValueError(f"dropout must be in [0, 1), got {dropout}")
    flat = [p for lp in layer_params for p in lp]
    widths = {lp[0].size(1) for lp in layer_params} | {lp[0].size(0) for lp in layer_params[1:]}
    if not has_bias and widths == {32}:
        if FORWARD_AGGREGATE_FIRST and aggregate_first and not x.requires_grad and (x.size(1) <= 4 or x.size(1) == 32):
            return _ResidualGCNStack32AT.apply(x, graph, pre, post, last_relu, dropout, *flat)
        if dropout > 0:
            return None
        return _ResidualGCNStack32.apply(x, graph, pre, post, last_relu, *flat)
    return _ResidualGCNStack.apply(x, graph, pre, post, has_bias, last_relu, dropout, *flat)
