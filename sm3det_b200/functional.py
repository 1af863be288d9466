"""autograd.Function wrappers: one per fused stage of the backbone, forward and hand-written backward.

Each Function only sequences C-ABI kernel calls (sm3det_b200.ops); tensors stay NHWC fp32 between
stages.  What each one replaces in the reference (mmrotate/models/backbones/convnext_moe.py):
  StemFn        dataset_stems['single'] + downsample_layers[0]            :783-791, :800-806
  DownsampleFn  Sequential(LayerNorm2d, Conv2d(2, stride 2))              :549-558, :806
  DenseBlockFn  ConvNeXtBlock._inner_forward with FFN                     :343-372, :397-405
  MoEBlockFn    ConvNeXtBlock._inner_forward with MoE_layer               :343-372, :226-293
  OutNormFn     norm{i}(x) channel_first incl. permute+contiguous         :811-817, :34-47
Backward follows SURVEY.md Appendix F (what autograd derives for the reference).

The only torch arithmetic left in this file is O(#parameters) glue on weight-sized tensors
(transposing 7x7 taps, flipping them for dgrad, multiplying a [C] vector by gamma).
"""
import torch
from torch.autograd import Function

from . import ops
from .ops import (EPI_AUXSTORE, EPI_COLSCALE, EPI_DGELU, EPI_GELU, EPI_RESID, EPI_ROWSCALE, LN_NCHW, LN_NHWC, LN_PATCH2)


def _zeros_like_param(p):
    return torch.zeros(p.shape, device=p.device, dtype=torch.float32)


def _taps(w):              # [C,1,ks,ks] -> [ks*ks][C]
    return w.reshape(w.shape[0], -1).t().contiguous()


def _taps_flipped(w):      # correlation taps for dgrad
    return w.flip(2, 3).reshape(w.shape[0], -1).t().contiguous()


@ops.captures_precision
class StemFn(Function):
    @staticmethod
    def forward(ctx, x, w, b, lnw, lnb, eps, ps):
        C0 = w.shape[0]
        wt = w.reshape(C0, -1).t().contiguous()
        train = any(ctx.needs_input_grad)
        x = x.contiguous().float()
        y, conv, stats = ops.stem_fwd(x, wt, b, lnw, lnb, eps, ps, save=train)
        if train:
            ctx.save_for_backward(x, conv, stats, lnw)
            ctx.ps = ps
            ctx.wshape = tuple(w.shape)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, conv, stats, lnw = ctx.saved_tensors
        dy = dy.contiguous()
        C0 = lnw.shape[0]
        T = conv.numel() // C0
        dlnw, dlnb = _zeros_like_param(lnw), _zeros_like_param(lnw)
        du = ops.layernorm_bwd(dy, conv, stats, lnw, dlnw, dlnb, tokens=T, C=C0)
        # weight gradient on the tensor cores: patches gathered once (im2col of the non-overlapping ps x ps patches, columns
        # ordered (kh, kw, ci), zero padded to a multiple of 32) and reduced over all tokens by the split-K GEMM -- 5x faster
        # than the SIMT stem_wgrad kernel at 1024^2 (0.25 vs 1.15 ms per step)
        N, Cin, H, W = x.shape
        ps = ctx.ps
        K = Cin * ps * ps
        Kp = (K + 31) // 32 * 32
        if C0 % 8 == 0:
            col, _, _ = ops.im2col(x, N=N, H=H, W=W, Cin=Cin, ks=ps, stride=ps, pad=0, Kp=Kp, nchw=True)
            dw2 = torch.zeros((C0, Kp), device=x.device, dtype=torch.float32)
            ops.linear_wgrad(du, col, dw2)
            db = torch.zeros((C0,), device=x.device, dtype=torch.float32)
            ops.colsum(du, db, rows=T, Cc=C0)
            dw = dw2[:, :K].reshape(C0, ps, ps, Cin).permute(0, 3, 1, 2).contiguous()
            return None, dw, db, dlnw, dlnb, None, None
        dwt = torch.zeros((K, C0), device=x.device, dtype=torch.float32)
        db = torch.zeros((C0,), device=x.device, dtype=torch.float32)
        ops.stem_wgrad(x, du, dwt, db, ctx.ps)
        dw = dwt.t().reshape(ctx.wshape).contiguous()
        return None, dw, db, dlnw, dlnb, None, None


@ops.captures_precision
class DownsampleFn(Function):
    @staticmethod
    def forward(ctx, x, lnw, lnb, w, b, eps):
        N, H, W, C = x.shape
        Co = w.shape[0]
        T = N * H * W
        train = any(ctx.needs_input_grad)
        xn = torch.empty((T // 4, 4 * C), device=x.device, dtype=torch.float32)
        _, stats = ops.layernorm_fwd(x, lnw, lnb, eps, tokens=T, C=C, out=xn, out_mode=LN_PATCH2, H=H, W=W,
                                     save_stats=train)
        w2 = w.permute(0, 2, 3, 1).reshape(Co, 4 * C).contiguous()      # [Co, (kh, kw, ci)]
        # w2 is a per-call re-ordered copy of the conv weight: split it once here (a few us) so both operands take the
        # bulk-copy main loop (4x the throughput of the in-kernel split on these shapes)
        y = ops.linear_fwd(xn, w2, b, packed=ops.pack_weight(w2, transposed=False))
        if train:
            ctx.save_for_backward(x, stats, xn, lnw, w2)
            ctx.dims = (N, H, W, C, Co)
        return y.view(N, H // 2, W // 2, Co)

    @staticmethod
    def backward(ctx, dy):
        x, stats, xn, lnw, w2 = ctx.saved_tensors
        N, H, W, C, Co = ctx.dims
        T = N * H * W
        dy2 = dy.contiguous().view(T // 4, Co)
        dxn = ops.linear_dgrad(dy2, w2, packed=ops.pack_weight(w2, transposed=True))
        dw2 = torch.zeros_like(w2)
        ops.linear_wgrad(dy2, xn, dw2)
        db = torch.zeros((Co,), device=x.device, dtype=torch.float32)
        ops.colsum(dy2, db, rows=T // 4, Cc=Co)
        dlnw, dlnb = _zeros_like_param(lnw), _zeros_like_param(lnw)
        dx = ops.layernorm_bwd(dxn, x, stats, lnw, dlnw, dlnb, tokens=T, C=C, in_mode=LN_PATCH2, H=H, W=W)
        dw = dw2.view(Co, 2, 2, C).permute(0, 3, 1, 2).contiguous()
        return dx.view(N, H, W, C), dlnw, dlnb, dw, db, None


@ops.captures_precision
class OutNormFn(Function):
    @staticmethod
    def forward(ctx, x, w, b, eps):
        N, H, W, C = x.shape
        T = N * H * W
        train = any(ctx.needs_input_grad)
        y = torch.empty((N, C, H, W), device=x.device, dtype=torch.float32)
        _, stats = ops.layernorm_fwd(x, w, b, eps, tokens=T, C=C, out=y, out_mode=LN_NCHW, H=H, W=W, save_stats=train)
        if train:
            ctx.save_for_backward(x, stats, w)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, stats, w = ctx.saved_tensors
        N, H, W, C = x.shape
        dw, db = _zeros_like_param(w), _zeros_like_param(w)
        dx = ops.layernorm_bwd(dy.contiguous(), x, stats, w, dw, db, tokens=N * H * W, C=C, in_mode=LN_NCHW, H=H, W=W)
        return dx.view(N, H, W, C), dw, db, None


def _block_front(x, dww, dwb, lnw, lnb, eps, train):
    N, H, W, C = x.shape
    u = ops.dwconv7(x, _taps(dww), dwb)
    v, stats = ops.layernorm_fwd(u, lnw, lnb, eps, tokens=N * H * W, C=C, save_stats=train)
    return u, v.view(N * H * W, C), stats


def _block_front_bwd(dv, dout, x, u, stats, dww, lnw):
    """LN backward -> depthwise dgrad (+ shortcut gradient) and the depthwise/LN parameter grads."""
    N, H, W, C = x.shape
    T = N * H * W
    dlnw, dlnb = _zeros_like_param(lnw), _zeros_like_param(lnw)
    du = ops.layernorm_bwd(dv, u, stats, lnw, dlnw, dlnb, tokens=T, C=C).view(N, H, W, C)
    dx = ops.dwconv7(du, _taps_flipped(dww), None, resid=dout)
    ddwt = torch.zeros((49, C), device=x.device, dtype=torch.float32)
    ddwb = torch.zeros((C,), device=x.device, dtype=torch.float32)
    ops.dwconv7_wgrad(x, du, ddwt, ddwb)
    ddww = ddwt.t().reshape(C, 1, 7, 7).contiguous()
    return dx, ddww, ddwb, dlnw, dlnb


@ops.captures_precision
class DenseBlockFn(Function):
    """Dense ConvNeXt block.  Narrow stages (ops.ffn_chunk: C <= 192) run the FFN forward as the fused tcgen05 kernel of
    csrc/ffn_fused.cu (GEMM1 -> GELU -> GEMM2 on chip; the hidden tensor is written once, as fp32 h, only when a backward
    follows).  The backward is the GEMM sequence (dgrad2 -> act_pack -> wgrads / dgrad1): fused recompute kernels for it
    were built and measured slower (narrow tcgen05 MMAs are paced by the 64-byte/clk operand fetch, not by N --
    profiles/r02_mma_microbench.txt).  Wider stages keep GEMM -> act_pack -> GEMM."""

    @staticmethod
    def forward(ctx, x, dww, dwb, lnw, lnb, w1, b1, w2, b2, gamma, row_scale, eps, packs):
        N, H, W, C = x.shape
        T = N * H * W
        # autograd.Function.forward runs with grad mode off and needs_input_grad reflects requires_grad only: the caller
        # says whether a backward can follow (it also chose which weight images to provide on that basis)
        train = any(ctx.needs_input_grad) and packs.get('grad', True)
        fused = packs.get('fused')
        # packs['shortcut'] = False: return the branch gamma * ffn(...) alone (ConvNeXt_DA gates it before the shortcut add)
        ctx.shortcut = packs.get('shortcut', True)
        resid = x.view(T, C) if ctx.shortcut else None
        if fused is not None:
            # LayerNorm writes the FFN's A-operand image directly (the separate split pass never exists); the fused kernel
            # keeps the hidden tensor on chip and, when a backward follows, stores the pre-activation h once for it
            u = ops.dwconv7(x, _taps(dww), dwb)
            v_img, v, stats = ops.layernorm_fwd_img(u, lnw, lnb, eps, tokens=T, C=C, save_stats=train, want_f32=train)
            res = ops.ffn_fused_fwd(v_img, packs['w1_c'][0], packs['w2_n'][0], b1, b2, T=T, C=C, chunk=fused['fwd'],
                                    gamma=gamma, row_scale=row_scale, resid=resid, want_aux=train, want_h=train)
            if train:
                ctx.save_for_backward(x, u, stats, v, res[2], res[1], dww, lnw, w1, w2, gamma, row_scale)
                ctx.packs = packs
            return res[0].view(N, H, W, C)
        u, v, stats = _block_front(x, dww, dwb, lnw, lnb, eps, train)
        # GEMM1 stores the pre-activation only; GELU runs in the HBM-bound act_pack kernel, which emits the result
        # directly as GEMM2's pre-split A operand (fp32 `a` never exists)
        h = ops.linear_fwd(v, w1, b1, packed=packs.get('w1'))
        a_k, _, _ = ops.act_pack(h, rows=T, width=4 * C, mode=ops.ACT_GELU, want_k=True)
        y2 = torch.empty((T, C), device=x.device, dtype=torch.float32) if train else None
        epi = (EPI_COLSCALE | (EPI_RESID if resid is not None else 0) | (EPI_ROWSCALE if row_scale is not None else 0)
               | (EPI_AUXSTORE if train else 0))
        out = ops.linear_fwd(None, w2, b2, rows=T, a_packed=a_k, epilogue=epi, aux_out=y2, col_scale=gamma,
                             row_scale=row_scale, resid=resid, packed=packs.get('w2'))
        if train:
            ctx.save_for_backward(x, u, stats, v, h, y2, dww, lnw, w1, w2, gamma, row_scale)
            ctx.packs = packs
        return out.view(N, H, W, C)

    @staticmethod
    def backward(ctx, dout):
        x, u, stats, v, h, y2, dww, lnw, w1, w2, gamma, rs = ctx.saved_tensors
        N, H, W, C = x.shape
        T = N * H * W
        dout = dout.contiguous()
        dz = dout.view(T, C)
        dev = x.device
        if rs is None:
            csum, dgamma = ops.colstat(dz, rows=T, Cc=C, y=y2)            # one pass: sum dz and sum dz * y2
        else:
            dgamma = torch.zeros((C,), device=dev, dtype=torch.float32)
            ops.colsum(dz, dgamma, rows=T, Cc=C, b=y2, row_scale=rs)
            csum = torch.zeros((C,), device=dev, dtype=torch.float32)
            ops.colsum(dz, csum, rows=T, Cc=C, row_scale=rs)
        db2 = csum * gamma
        w2g = ops.scale_rows(w2, row_scale=gamma)                   # gamma[c] * W2[c, :]
        da = ops.linear_dgrad(dz, w2g, epilogue=(EPI_ROWSCALE if rs is not None else 0), row_scale=rs,
                              packed=ops.pack_weight(w2g, transposed=True))
        # dh = da * gelu'(h) goes straight into the two operand images (dgrad1's A, wgrad1's A) + db1 column sums
        db1 = torch.zeros((4 * C,), device=dev, dtype=torch.float32)
        # one pass over h: dh = da * gelu'(h) as dgrad1's / wgrad1's operands (+ db1) and a = gelu(h) as wgrad2's operand
        dh_k, dh_mn, a_mn = ops.act_pack(h, rows=T, width=4 * C, mode=ops.ACT_BWD, da=da, want_k=True, mn_tile=128,
                                      mn_tile2=ops._pick_bn(4 * C), colsum=db1)
        del da
        dzs = dz if rs is None else ops.scale_rows(dz, row_scale=rs)
        dw2 = torch.zeros_like(w2)
        ops.linear_wgrad(dzs, None, dw2, rows=T, row_scale=gamma, x_packed=a_mn)
        del a_mn
        dw1 = torch.zeros_like(w1)
        ops.linear_wgrad(None, v, dw1, rows=T, dy_packed=dh_mn)
        dv = ops.linear_dgrad(None, w1, rows=T, a_packed=dh_k, packed=ctx.packs.get('w1_t'))
        dx, ddww, ddwb, dlnw, dlnb = _block_front_bwd(dv, dout if ctx.shortcut else None, x, u, stats, dww, lnw)
        return dx, ddww, ddwb, dlnw, dlnb, dw1, db1, dw2, db2, dgamma, None, None, None


def stack_expert_params(params):
    """Make E same-shaped parameters views of one contiguous [E, ...] buffer (grouped-GEMM layout).

    Parameter objects (and therefore optimizer state, named_parameters() and state_dict keys) are
    untouched; only ``.data`` is re-pointed.  No-op when they are already adjacent in memory.
    """
    base = params[0]
    step = base.numel() * base.element_size()
    if all(p.is_contiguous() and p.data_ptr() == base.data_ptr() + i * step for i, p in enumerate(params)):
        return
    with torch.no_grad():
        flat = torch.stack([p.data for p in params]).contiguous()
        for i, p in enumerate(params):
            p.data = flat[i]


def gating_noise(layer, T, device):
    """[T, E] gating noise of a noisy-gating MoE layer in training, else None (tests inject ``_injected_noise``)."""
    if not (layer.noisy_gating and layer.training):
        return None
    noise = getattr(layer, '_injected_noise', None)
    if noise is None:
        noise = torch.randn((T, layer.num_experts), device=device, dtype=torch.float32)
    return noise.to(device, torch.float32).contiguous()


def drop_path_row_scale(block, x):
    """timm DropPath as a per-token scale of NHWC x (per-sample Bernoulli(keep) / keep), None when inactive.
    Tests inject the per-sample mask as ``_injected_drop_mask``."""
    if block.drop_path_rate == 0. or not block.training:
        return None
    keep = 1.0 - block.drop_path_rate
    N, H, W, _ = x.shape
    mask = getattr(block, '_injected_drop_mask', None)
    if mask is None:
        mask = x.new_empty((N,)).bernoulli_(keep)
        if keep > 0.0:
            mask = mask / keep
    return mask.to(x.device, torch.float32).repeat_interleave(H * W).contiguous()


def route(v, wp, bp, sim, tau, w_noise, noise, *, T, C, E, k, save):
    """Router -> plan -> slot assignment of one MoE layer: (r, plan, slot_of, pair_token)."""
    r = ops.moe_router(v, wp, bp, sim, tau, T=T, Cc=C, E=E, k=k, w_noise=w_noise, noise=noise, save=save)
    plan = ops.moe_plan(r['partials'], T=T, E=E, k=k)
    slot_of, pair_token = ops.moe_assign(r['top_idx'], plan, T=T, E=E, k=k)
    return r, plan, slot_of, pair_token


ROUTER_SAVED = 13      # number of tensors router_saved returns


def router_saved(r, plan, sim, tau, noise, w_noise):
    """The tensors router_backward needs, in its order; top_idx and top_gate come first (combine backward uses them)."""
    return (r['top_idx'], r['top_gate'], r['p'], sim, tau, r['logits'], plan['importance'], noise, r['sigma'],
            r['top_vals'], r['top_idx_m'], plan['load'], w_noise)


def router_backward(saved, v, wp, dgate, dloss, wp_t=None):
    """(dv_r, dwp, dbp, dsim, dtau, dwn) of the router that saw the rows v [T, C]; ``saved`` is router_saved(...).
    The gates depend on w_noise whenever noise was drawn, also for k == E.  Without noise dwn is zero (DDP wants a
    gradient for every parameter), None if the layer has no w_noise."""
    top_idx, top_gate, p, sim, tau, logits, importance, noise, sigma, top_vals, top_idx_m, load, w_noise = saved
    T, C = v.shape
    P, E = sim.shape
    k = top_idx.shape[1]
    dev = v.device
    dtau = torch.zeros((1,), device=dev, dtype=torch.float32)
    dsim = torch.zeros((P, E), device=dev, dtype=torch.float32)
    lscale = dloss.reshape(1).contiguous().float()
    noisy = None if noise is None else dict(noise=noise, sigma=sigma, top_vals=top_vals, top_idx_m=top_idx_m, load=load)
    dp, dr = ops.moe_router_bwd(p, sim, tau, top_idx, top_gate, dgate, logits, importance, lscale, dsim, dtau, T=T,
                                E=E, k=k, noisy=noisy)
    dwp = torch.zeros_like(wp)
    ops.linear_wgrad(dp, v, dwp)
    dbp = torch.zeros((P,), device=dev, dtype=torch.float32)
    ops.colsum(dp, dbp, rows=T, Cc=P)
    dv_r = ops.linear_dgrad(dp, wp, packed=wp_t)
    dwn = None
    if noise is not None:
        # r = v @ w_noise is an [T,C]x[C,E] product with E < 32: run it as a 32-wide zero-padded GEMM pair
        wn_t = torch.zeros((32, C), device=dev, dtype=torch.float32)
        wn_t[:E] = w_noise.t()
        dwn_t = torch.zeros((32, C), device=dev, dtype=torch.float32)
        ops.linear_wgrad(dr, v, dwn_t)                             # [32,C] = dr^T v
        dwn = dwn_t[:E].t().contiguous()
        dv_r = ops.linear_dgrad(dr, wn_t, epilogue=EPI_RESID, resid=dv_r)
    elif w_noise is not None:
        dwn = torch.zeros((C, E), device=dev, dtype=torch.float32)
    return dv_r, dwp, dbp, dsim, dtau, dwn


def expert_ffn_fwd(a, w1, b1, w2, b2, packs, *, rows, grouped, row_index=None, out=None):
    """Grouped two-GEMM experts over ``rows`` expert-sorted rows: h = a[row_index] w1^T + b1 (no row_index: a is in
    expert order already), o = gelu(h) w2^T + b2 (into ``out`` when given).  w1 .. b2 are the first expert's stacked
    parameters (stack_expert_params).  Returns (h, o)."""
    C = a.shape[1]
    h = ops.linear_fwd(a, w1, b1, row_index=row_index, rows=rows, grouped=grouped, w_group_stride=4 * C * C,
                       bias_group_stride=4 * C, packed=packs.get('w1'))
    a_k, _, _ = ops.act_pack(h, rows=rows, width=4 * C, mode=ops.ACT_GELU, want_k=True, live_tiles=grouped[1])
    o = ops.linear_fwd(None, w2, b2, rows=rows, a_packed=a_k, grouped=grouped, w_group_stride=4 * C * C,
                       bias_group_stride=C, packed=packs.get('w2'), out=out)
    return h, o


def expert_ffn_bwd(d_o, h, a, w1, w2, packs, *, rows, grouped, segs, groups, row_index=None, dxp=None):
    """Backward of expert_ffn_fwd: (dxp, dw1s, db1s, dw2s, db2s), weight gradients stacked over ``groups`` experts.
    dxp (the given buffer, or a new one) is written at every live row; padding rows are never read."""
    C = a.shape[1]
    dev = d_o.device
    da = ops.linear_dgrad(d_o, w2, grouped=grouped, w_group_stride=4 * C * C, packed=packs.get('w2_t'))
    db1s = torch.zeros((groups, 4 * C), device=dev, dtype=torch.float32)
    # one pass over h: dh = da * gelu'(h) as dgrad1's / wgrad1's operands (+ db1) and a = gelu(h) as wgrad2's operand
    dh_k, dh_mn, a_mn = ops.act_pack(h, rows=rows, width=4 * C, mode=ops.ACT_BWD, da=da, want_k=True, mn_tile=128,
                                     mn_tile2=ops._pick_bn(4 * C), colsum=db1s, live_tiles=grouped[1],
                                     tile_group=grouped[0])
    del da
    dw2s = torch.zeros((groups, C, 4 * C), device=dev, dtype=torch.float32)
    ops.linear_wgrad(d_o, None, dw2s, rows=rows, segs=segs, num_groups=groups, x_packed=a_mn)
    del a_mn
    db2s = torch.zeros((groups, C), device=dev, dtype=torch.float32)
    ops.colsum(d_o, db2s, rows=rows, Cc=C, segs=segs, groups=groups)
    dw1s = torch.zeros((groups, 4 * C, C), device=dev, dtype=torch.float32)
    ops.linear_wgrad(None, a, dw1s, rows=rows, x_row_index=row_index, segs=segs, num_groups=groups, dy_packed=dh_mn)
    if dxp is None:
        dxp = torch.empty((rows, C), device=dev, dtype=torch.float32)
    ops.linear_dgrad(None, w1, rows=rows, a_packed=dh_k, out=dxp, grouped=grouped, w_group_stride=4 * C * C,
                     packed=packs.get('w1_t'))
    return dxp, dw1s, db1s, dw2s, db2s


@ops.captures_precision
class MoEBlockFn(Function):
    """x -> dwconv -> LN -> router/plan/assign -> grouped expert GEMMs -> combine (+gamma, +shortcut)."""

    @staticmethod
    def forward(ctx, x, dww, dwb, lnw, lnb, gamma, wp, bp, sim, tau, w_noise, row_scale, noise, eps, E, k, record, packs,
                *experts):
        N, H, W, C = x.shape
        T = N * H * W
        w1s, b1s, w2s, b2s = experts[0:E], experts[E:2 * E], experts[2 * E:3 * E], experts[3 * E:4 * E]
        train = any(ctx.needs_input_grad)
        u, v, stats = _block_front(x, dww, dwb, lnw, lnb, eps, train)
        r, plan, slot_of, pair_token = route(v, wp, bp, sim, tau, w_noise, noise, T=T, C=C, E=E, k=k, save=train)
        R = plan['max_rows']
        h, o = expert_ffn_fwd(v, w1s[0], b1s[0], w2s[0], b2s[0], packs, rows=R,
                              grouped=(plan['tile_group'], plan['num_m_tiles']), row_index=pair_token)
        ctx.shortcut = packs.get('shortcut', True)
        out, y = ops.moe_combine(o, slot_of, r['top_idx'], r['top_gate'], gamma, x.view(T, C) if ctx.shortcut else None,
                                 row_scale, T=T, Cc=C, k=k, want_y=record is not None)
        if record is not None:
            record.append(dict(v=v, top_idx=r['top_idx'], top_gate=r['top_gate'], importance=plan['importance'],
                               load=plan['load'], loss=plan['loss'], y=y, counts=plan['counts']))
        if train:
            ctx.save_for_backward(*router_saved(r, plan, sim, tau, noise, w_noise), x, u, stats, v, h, o, dww, lnw, gamma,
                                  wp, row_scale, slot_of, pair_token, plan['seg_begin'], plan['seg_end'],
                                  plan['tile_group'], plan['num_m_tiles'], w1s[0], w2s[0])
            ctx.E, ctx.k, ctx.R = E, k, R
            ctx.packs = packs
        return out.view(N, H, W, C), plan['loss'].reshape(())

    @staticmethod
    def backward(ctx, dout, dloss):
        saved = ctx.saved_tensors
        router = saved[:ROUTER_SAVED]
        (x, u, stats, v, h, o, dww, lnw, gamma, wp, rs, slot_of, pair_token, seg_begin, seg_end, tile_group, num_m_tiles,
         w1, w2) = saved[ROUTER_SAVED:]
        top_idx, top_gate = router[:2]
        E, k, R = ctx.E, ctx.k, ctx.R
        N, H, W, C = x.shape
        T = N * H * W
        dev = x.device
        dout = dout.contiguous()
        dz = dout.view(T, C)
        # combine / layer scale / shortcut
        d_o = torch.zeros((R, C), device=dev, dtype=torch.float32)
        dgamma = torch.zeros((C,), device=dev, dtype=torch.float32)
        dgate = ops.moe_combine_bwd(dz, o, slot_of, top_idx, top_gate, gamma, rs, d_o, dgamma, T=T, Cc=C, k=k)
        # experts (grouped over the padded expert segments)
        dxp, dw1s, db1s, dw2s, db2s = expert_ffn_bwd(d_o, h, v, w1, w2, ctx.packs, rows=R, grouped=(tile_group, num_m_tiles),
                                                     segs=(seg_begin, seg_end), groups=E, row_index=pair_token)
        dv_r, dwp, dbp, dsim, dtau, dwn = router_backward(router, v, wp, dgate, dloss, ctx.packs.get('wp_t'))
        dv = ops.gather_sum(dxp, slot_of, dv_r, T=T, Cc=C, k=k)
        dx, ddww, ddwb, dlnw, dlnb = _block_front_bwd(dv, dout if ctx.shortcut else None, x, u, stats, dww, lnw)
        grads_e = [dw1s[e] for e in range(E)] + [db1s[e] for e in range(E)] + [dw2s[e] for e in range(E)] + \
                  [db2s[e] for e in range(E)]
        return (dx, ddww, ddwb, dlnw, dlnb, dgamma, dwp, dbp, dsim, dtau, dwn, None, None, None, None, None, None, None,
                *grads_e)


@ops.captures_precision
class DAGateFn(Function):
    """ConvNeXt_DA block tail (convnext_moe_DA.py:400-401): out = shortcut + row_scale * s[n, c] * y  with y the gamma-scaled
    FFN branch [N,H,W,C] and s = DALayer's per-sample channel gate [N,C]; also returns nothing else -- the squeeze
    (per-sample mean of y) is SampleMeanFn.  Per sample one `affine` launch (N is the per-GPU batch)."""

    @staticmethod
    def forward(ctx, y, x, s, row_scale):
        N, H, W, C = y.shape
        y, x = y.contiguous(), x.contiguous()
        hw = H * W
        out = torch.empty_like(x)
        # per-sample scale vector: s[n] (* the sample's drop-path factor: row_scale is constant over a sample's tokens)
        sc = s if row_scale is None else s * row_scale.view(N, hw)[:, :1]
        sc = sc.contiguous()
        for n in range(N):
            ops.affine(y[n].view(hw, C), a1=sc[n], add=x[n].view(hw, C), out=out[n].view(hw, C))
        ctx.save_for_backward(y, sc, s, row_scale)
        return out

    @staticmethod
    def backward(ctx, d):
        y, sc, s, rs = ctx.saved_tensors
        N, H, W, C = y.shape
        hw = H * W
        d = d.contiguous()
        dy = torch.empty_like(y)
        dsc = torch.zeros((N, C), device=y.device, dtype=torch.float32)
        for n in range(N):
            ops.affine(d[n].view(hw, C), a1=sc[n], out=dy[n].view(hw, C))
            ops.colsum(d[n].view(hw, C), dsc[n], rows=hw, Cc=C, b=y[n].view(hw, C))       # sum_hw d * y
        ds = dsc if rs is None else dsc * rs.view(N, hw)[:, :1]
        return dy, d, ds, None


@ops.captures_precision
class SampleMeanFn(Function):
    """DALayer's squeeze: AdaptiveAvgPool2d(1) over an NHWC tensor -> [N, C]."""

    @staticmethod
    def forward(ctx, y):
        N, H, W, C = y.shape
        y = y.contiguous()
        m = torch.zeros((N, C), device=y.device, dtype=torch.float32)
        for n in range(N):
            ops.colsum(y[n].view(H * W, C), m[n], rows=H * W, Cc=C)
        ctx.shape = (N, H, W, C)
        return m / float(H * W)

    @staticmethod
    def backward(ctx, dm):
        N, H, W, C = ctx.shape
        return (dm / float(H * W)).view(N, 1, 1, C).expand(N, H, W, C).contiguous()
