"""autograd.Function wrappers of the LSKNet-MoE backbone (BASELINE config 5): forward and hand-written backward.

Each Function only sequences C-ABI kernel calls (sm3det_b200.ops); activations stay NHWC fp32.  What each one
replaces in the reference (mmrotate/models/backbones/lsk_moe.py):
  BatchNormFn    nn.BatchNorm2d / SyncBatchNorm built by build_norm_layer        :369-374, :407-410, :692-695
  LinearFn       every 1x1 nn.Conv2d (proj_1/2, conv1/2, conv, fc1/fc2) (+GELU)  :324-327, :351-354, :293-298
  DWConvFn       depthwise 5x5, 7x7 dilation 3, 3x3                              :322-323, :583
  GeluFn         Mlp.act                                                         :310
  LSKSelectFn    mean/max -> conv_squeeze -> sigmoid -> weighted sum             :335-341
  MulFn          x * attn, dropout masks                                         :343, :311, :316
  AxpyFn         layer-scale * branch + shortcut                                 :362, :388-395
  PatchEmbedFn   OverlapPatchEmbed.proj (7x7/s4 stem, 3x3/s2)                    :405-406, :689-691
  MoELinearFn    MoE_layer.forward with single-Conv2d experts + SparseDispatcher :195-273
Remaining torch arithmetic is O(#channels) glue on [C]-sized vectors (BN scale/shift, running statistics).
"""
import torch
import torch.distributed as dist
from torch.autograd import Function

from . import ops
from .functional import ROUTER_SAVED, _taps, _taps_flipped, route, router_backward, router_saved
from .ops import EPI_GELU


AMAX_RECORD = None   # parity tests set this to a list: LSKSelectFn appends the channel argmax [T] of every LSKblock (forward order)


def _sync_active(sync):
    return bool(sync) and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1


def bn_batch_stats(s1, s2, n, running_mean, sync, group=None):
    """(mean, biased var, n) of a (Sync)BatchNorm from the per-rank shifted sums s1 = sum(x - running_mean),
    s2 = sum((x - running_mean)^2) over n local rows.  With ``sync`` the three are all-reduced first: the shift is the
    running mean, identical on every rank, so the sums simply add.  Pure [C]-sized glue (CPU-testable, gloo).  With ``sync``
    the returned n is a 0-dim tensor that stays on the device: no host read-back per normalisation layer."""
    C = s1.numel()
    if _sync_active(sync):
        st = torch.cat([s1, s2, torch.full((1,), float(n), device=s1.device, dtype=s1.dtype)])
        dist.all_reduce(st, group=group)
        s1, s2, n = st[:C], st[C:2 * C], st[2 * C]
    else:
        n = float(n)
    d = s1 / n
    return running_mean + d, (s2 / n - d * d).clamp_min_(0.0), n


@ops.captures_precision
class BatchNormFn(Function):
    """y = BN(x) over all tokens (and all ranks when ``sync``); updates the running buffers in training mode."""

    @staticmethod
    def forward(ctx, x, weight, bias, running_mean, running_var, train, momentum, eps, sync):
        C = x.shape[-1]
        rows = x.numel() // C
        x = x.contiguous()
        if train:
            # one pass, data shifted by the running mean (identical on every rank): s1 = sum(x-rm), s2 = sum (x-rm)^2
            s1, s2 = ops.colstat(x, rows=rows, Cc=C, sh1=running_mean)
            mean, var, n = bn_batch_stats(s1, s2, float(rows), running_mean, sync)
            rstd = torch.rsqrt(var + eps)
            with torch.no_grad():
                running_mean.mul_(1 - momentum).add_(mean, alpha=momentum)
                unbias = n / torch.clamp(n - 1.0, min=1.0) if torch.is_tensor(n) else n / max(n - 1.0, 1.0)
                running_var.mul_(1 - momentum).add_(var * unbias, alpha=momentum)
        else:
            mean, rstd, n = running_mean, torch.rsqrt(running_var + eps), float(rows)
        scale = (weight * rstd).contiguous()
        shift = (bias - mean * scale).contiguous()
        y = ops.affine(x, a1=scale, b=shift)
        if any(ctx.needs_input_grad):
            ctx.save_for_backward(x, weight, mean.contiguous(), rstd.contiguous())
            ctx.train, ctx.n, ctx.sync = train, n, sync
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight, mean, rstd = ctx.saved_tensors
        C = x.shape[-1]
        rows = x.numel() // C
        dy = dy.contiguous()
        s1, s2 = ops.colstat(dy, rows=rows, Cc=C, y=x, sh2=mean, sc2=rstd)      # sum dy, sum dy * xhat
        dw, db = s2.clone(), s1.clone()
        A = (weight * rstd).contiguous()
        if ctx.train:
            if _sync_active(ctx.sync):
                st = torch.cat([s1, s2])
                dist.all_reduce(st)
                s1, s2 = st[:C], st[C:]
            Bc = (-(A * rstd) * (s2 / ctx.n)).contiguous()
            D = (-(A * (s1 / ctx.n)) - Bc * mean).contiguous()
            dx = ops.affine(dy, a1=A, x2=x, a2=Bc, b=D)
        else:
            dx = ops.affine(dy, a1=A)
        return dx, dw, db, None, None, None, None, None, None


@ops.captures_precision
class LinearFn(Function):
    """y[T,N] = act(x[T,K] @ w[N,K]^T + b); w may be a 1x1 conv weight [N,K,1,1]."""

    @staticmethod
    def forward(ctx, x, w, b, gelu):
        lead = x.shape[:-1]
        K = x.shape[-1]
        x2 = x.contiguous().view(-1, K)
        w2 = w.view(w.shape[0], K)
        train = any(ctx.needs_input_grad)
        h = torch.empty((x2.shape[0], w2.shape[0]), device=x.device, dtype=torch.float32) if (gelu and train) else None
        # weights are split per call (a few us; 1x1 conv weights are small) so both operands take the bulk-copy main loop
        y = ops.linear_fwd(x2, w2, b, epilogue=EPI_GELU if gelu else 0, aux_out=h, packed=ops.pack_weight(w2, transposed=False))
        if train:
            ctx.save_for_backward(x2, w2, h)
            ctx.wshape, ctx.gelu, ctx.has_b = tuple(w.shape), gelu, b is not None
        return y.view(*lead, w2.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, w2, h = ctx.saved_tensors
        N, K = w2.shape
        T = x2.shape[0]
        dy2 = dy.contiguous().view(T, N)
        db = torch.zeros((N,), device=dy.device, dtype=torch.float32) if ctx.has_b else None
        if ctx.gelu:
            _, _, dy2 = ops.act_pack(h, rows=T, width=N, mode=ops.ACT_DGELU, da=dy2, want_f32=True, colsum=db)
        elif db is not None:
            ops.colsum(dy2, db, rows=T, Cc=N)
        dw = torch.zeros((N, K), device=dy.device, dtype=torch.float32)
        ops.linear_wgrad(dy2, x2, dw)
        dx = ops.linear_dgrad(dy2, w2, packed=ops.pack_weight(w2, transposed=True)) if ctx.needs_input_grad[0] else None
        return (None if dx is None else dx.view(*dy.shape[:-1], K)), dw.view(ctx.wshape), db, None


@ops.captures_precision
class DWConvFn(Function):
    @staticmethod
    def forward(ctx, x, w, b, ks, dil):
        x = x.contiguous()
        y = ops.dwconv(x, _taps(w), b, ks=ks, dil=dil)
        if any(ctx.needs_input_grad):
            ctx.save_for_backward(x, w)
            ctx.ks, ctx.dil = ks, dil
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        C = x.shape[-1]
        dy = dy.contiguous()
        dx = ops.dwconv(dy, _taps_flipped(w), None, ks=ctx.ks, dil=ctx.dil)
        dwt = torch.zeros((ctx.ks * ctx.ks, C), device=x.device, dtype=torch.float32)
        db = torch.zeros((C,), device=x.device, dtype=torch.float32)
        ops.dwconv_wgrad(x, dy, dwt, db, ks=ctx.ks, dil=ctx.dil)
        return dx, dwt.t().reshape(w.shape).contiguous(), db, None, None


@ops.captures_precision
class GeluFn(Function):
    @staticmethod
    def forward(ctx, h):
        h = h.contiguous()
        W = h.shape[-1]
        _, _, y = ops.act_pack(h.view(-1, W), rows=h.numel() // W, width=W, mode=ops.ACT_GELU, want_f32=True)
        if ctx.needs_input_grad[0]:
            ctx.save_for_backward(h)
        return y.view(h.shape)

    @staticmethod
    def backward(ctx, dy):
        (h,) = ctx.saved_tensors
        W = h.shape[-1]
        _, _, dh = ops.act_pack(h.view(-1, W), rows=h.numel() // W, width=W, mode=ops.ACT_DGELU,
                                da=dy.contiguous().view(-1, W), want_f32=True)
        return dh.view(h.shape)


@ops.captures_precision
class LSKSelectFn(Function):
    """attn1*sig0 + attn2*sig1 with sig = sigmoid(conv_squeeze([mean_c, max_c] of cat(attn1, attn2)))."""

    @staticmethod
    def forward(ctx, a1, a2, wsq, bsq):
        N, H, W, Ch = a1.shape
        T = N * H * W
        a1, a2 = a1.contiguous(), a2.contiguous()
        train = any(ctx.needs_input_grad)
        agg, amax = ops.lsk_agg(a1, a2, T=T, Ch=Ch, want_idx=train or AMAX_RECORD is not None)
        if AMAX_RECORD is not None:
            AMAX_RECORD.append(amax)
        sig = ops.conv7_c2(agg, wsq.contiguous(), bsq, N=N, H=H, W=W, act=1)
        out = ops.lsk_mix(a1, a2, sig, T=T, Ch=Ch)
        if train:
            ctx.save_for_backward(a1, a2, agg, amax, sig, wsq)
        return out.view(N, H, W, Ch)

    @staticmethod
    def backward(ctx, dout):
        a1, a2, agg, amax, sig, wsq = ctx.saved_tensors
        N, H, W, Ch = a1.shape
        T = N * H * W
        dout = dout.contiguous()
        dpre = ops.lsk_mix_bwd_sig(dout, a1, a2, sig, T=T, Ch=Ch)
        dagg = ops.conv7_c2(dpre, wsq.flip(2, 3).transpose(0, 1).contiguous(), None, N=N, H=H, W=W, act=0)
        dw = torch.zeros((2, 2, 7, 7), device=dout.device, dtype=torch.float32)
        db = torch.zeros((2,), device=dout.device, dtype=torch.float32)
        ops.conv7_c2_wgrad(agg, dpre, dw, db, N=N, H=H, W=W)
        da1, da2 = ops.lsk_mix_bwd_in(dout, sig, dagg, amax, T=T, Ch=Ch)
        return da1.view(a1.shape), da2.view(a2.shape), dw, db


@ops.captures_precision
class MulFn(Function):
    @staticmethod
    def forward(ctx, a, b):
        a, b = a.contiguous(), b.contiguous()
        ctx.save_for_backward(a, b)
        return ops.mul(a, b)

    @staticmethod
    def backward(ctx, d):
        a, b = ctx.saved_tensors
        d = d.contiguous()
        da = ops.mul(d, b) if ctx.needs_input_grad[0] else None
        db = ops.mul(d, a) if ctx.needs_input_grad[1] else None
        return da, db


@ops.captures_precision
class DropoutFn(Function):
    """nn.Dropout with a counter-based mask: forward and backward are the same kernel with the same seed."""

    @staticmethod
    def forward(ctx, x, p, seed):
        ctx.p, ctx.seed = p, seed
        return ops.dropout(x.contiguous(), p, seed)

    @staticmethod
    def backward(ctx, d):
        return ops.dropout(d.contiguous(), ctx.p, ctx.seed), None, None


@ops.captures_precision
class AxpyFn(Function):
    """out = a[c] * y * row_scale[t] + x   (a = layer scale or None, row_scale = drop-path mask or None)."""

    @staticmethod
    def forward(ctx, y, x, a, row_scale):
        y, x = y.contiguous(), x.contiguous()
        ys = y if row_scale is None else ops.scale_rows(y, row_scale=row_scale)
        out = ops.affine(ys, a1=a, add=x)
        ctx.save_for_backward(ys if a is not None else None, a, row_scale)
        return out

    @staticmethod
    def backward(ctx, d):
        ys, a, rs = ctx.saved_tensors
        d = d.contiguous()
        C = d.shape[-1]
        da = None
        if a is not None:
            da = torch.zeros((C,), device=d.device, dtype=torch.float32)
            ops.colsum(d, da, rows=d.numel() // C, Cc=C, b=ys)
        dy = d if (a is None and rs is None) else ops.scale_rows(d, row_scale=rs, col_scale=a)
        return dy, d, da, None


@ops.captures_precision
class PatchEmbedFn(Function):
    """Conv2d(ks, stride, padding=ks//2) as im2col + tcgen05 GEMM.  x: NCHW (network input) or NHWC; out NHWC."""

    @staticmethod
    def forward(ctx, x, w, b, stride, nchw):
        Co, Ci, ks, _ = w.shape
        x = x.contiguous().float()
        if nchw:
            N, _, H, W = x.shape
        else:
            N, H, W, _ = x.shape
        K = ks * ks * Ci
        Kp = (K + 31) // 32 * 32
        col, Ho, Wo = ops.im2col(x, N=N, H=H, W=W, Cin=Ci, ks=ks, stride=stride, pad=ks // 2, Kp=Kp, nchw=nchw)
        w2 = torch.zeros((Co, Kp), device=w.device, dtype=torch.float32)
        w2[:, :K] = w.permute(0, 2, 3, 1).reshape(Co, K)
        y = ops.linear_fwd(col, w2, b, packed=ops.pack_weight(w2, transposed=False))
        if any(ctx.needs_input_grad):
            ctx.save_for_backward(x, w2)
            ctx.geom = (N, H, W, Ci, Co, ks, stride, K, Kp, nchw, Ho, Wo)
        return y.view(N, Ho, Wo, Co)

    @staticmethod
    def backward(ctx, dy):
        x, w2 = ctx.saved_tensors
        N, H, W, Ci, Co, ks, stride, K, Kp, nchw, Ho, Wo = ctx.geom
        T = N * Ho * Wo
        dy2 = dy.contiguous().view(T, Co)
        col, _, _ = ops.im2col(x, N=N, H=H, W=W, Cin=Ci, ks=ks, stride=stride, pad=ks // 2, Kp=Kp, nchw=nchw)
        dw2 = torch.zeros((Co, Kp), device=dy.device, dtype=torch.float32)
        ops.linear_wgrad(dy2, col, dw2)
        del col
        db = torch.zeros((Co,), device=dy.device, dtype=torch.float32)
        ops.colsum(dy2, db, rows=T, Cc=Co)
        dx = None
        if ctx.needs_input_grad[0]:
            dcol = ops.linear_dgrad(dy2, w2, packed=ops.pack_weight(w2, transposed=True))
            dx = ops.col2im(dcol, N=N, H=H, W=W, Cin=Ci, ks=ks, stride=stride, pad=ks // 2, Kp=Kp, nchw=nchw)
        dw = dw2[:, :K].reshape(Co, ks, ks, Ci).permute(0, 3, 1, 2).contiguous()
        return dx, dw, db, None, None


@ops.captures_precision
class MoELinearFn(Function):
    """LSKNet MoE layer: router -> plan -> grouped expert GEMM (single Conv2d(in,out,1) per expert, dispatch gather
    fused into the A-operand load) -> deterministic combine (x gamma + resid when given)."""

    @staticmethod
    def forward(ctx, x, wp, bp, sim, tau, w_noise, noise, gamma, resid, row_scale, E, k, record, *experts):
        Cin = x.shape[-1]
        lead = x.shape[:-1]
        x2 = x.contiguous().view(-1, Cin)
        T = x2.shape[0]
        ws, bs = experts[:E], experts[E:]
        Cout = ws[0].shape[0]
        train = any(ctx.needs_input_grad)
        r, plan, slot_of, pair_token = route(x2, wp, bp, sim, tau, w_noise, noise, T=T, C=Cin, E=E, k=k, save=train)
        R = plan['max_rows']
        grouped = (plan['tile_group'], plan['num_m_tiles'])
        w0 = ws[0].view(Cout, Cin)
        o = torch.zeros((R, Cout), device=x.device, dtype=torch.float32)
        ops.linear_fwd(x2, w0, bs[0], out=o, row_index=pair_token, rows=R, grouped=grouped, w_group_stride=Cout * Cin,
                       bias_group_stride=Cout)
        res2 = None if resid is None else resid.contiguous().view(T, Cout)
        out, y = ops.moe_combine(o, slot_of, r['top_idx'], r['top_gate'], gamma, res2, row_scale, T=T, Cc=Cout, k=k,
                                 want_y=record is not None)
        if record is not None:
            record.append(dict(x=x2, top_idx=r['top_idx'], top_gate=r['top_gate'], importance=plan['importance'],
                               load=plan['load'], loss=plan['loss'], y=y, counts=plan['counts']))
        if train:
            ctx.save_for_backward(*router_saved(r, plan, sim, tau, noise, w_noise), x2, o, wp, gamma, row_scale, slot_of,
                                  pair_token, plan['seg_begin'], plan['seg_end'], plan['tile_group'], plan['num_m_tiles'],
                                  w0)
            ctx.E, ctx.k, ctx.R, ctx.lead = E, k, R, tuple(lead)
            ctx.wshape = tuple(ws[0].shape)
            ctx.has_resid = resid is not None
        return out.view(*lead, Cout), plan['loss'].reshape(())

    @staticmethod
    def backward(ctx, dout, dloss):
        saved = ctx.saved_tensors
        router = saved[:ROUTER_SAVED]
        (x2, o, wp, gamma, rs, slot_of, pair_token, seg_begin, seg_end, tile_group, num_m_tiles,
         w0) = saved[ROUTER_SAVED:]
        top_idx, top_gate = router[:2]
        E, k, R = ctx.E, ctx.k, ctx.R
        T, Cin = x2.shape
        Cout = w0.shape[0]
        dev = x2.device
        dz = dout.contiguous().view(T, Cout)
        grouped, segs = (tile_group, num_m_tiles), (seg_begin, seg_end)
        d_o = torch.zeros((R, Cout), device=dev, dtype=torch.float32)
        dgamma = None if gamma is None else torch.zeros((Cout,), device=dev, dtype=torch.float32)
        dgate = ops.moe_combine_bwd(dz, o, slot_of, top_idx, top_gate, gamma, rs, d_o, dgamma, T=T, Cc=Cout, k=k)
        dws = torch.zeros((E, Cout, Cin), device=dev, dtype=torch.float32)
        ops.linear_wgrad(d_o, x2, dws, rows=R, x_row_index=pair_token, segs=segs, num_groups=E)
        dbs = torch.zeros((E, Cout), device=dev, dtype=torch.float32)
        ops.colsum(d_o, dbs, rows=R, Cc=Cout, segs=segs, groups=E)
        dxp = torch.zeros((R, Cin), device=dev, dtype=torch.float32)
        ops.linear_dgrad(d_o, w0, out=dxp, grouped=grouped, w_group_stride=Cout * Cin)
        dx_r, dwp, dbp, dsim, dtau, dwn = router_backward(router, x2, wp, dgate, dloss)
        dx = ops.gather_sum(dxp, slot_of, dx_r, T=T, Cc=Cin, k=k)
        dresid = dout if ctx.has_resid else None
        grads_e = [dws[e].view(ctx.wshape) for e in range(E)] + [dbs[e] for e in range(E)]
        return (dx.view(*ctx.lead, Cin), dwp, dbp, dsim, dtau, dwn, None, dgamma, dresid, None, None, None, None, *grads_e)
