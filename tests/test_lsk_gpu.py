"""GPU parity of the LSKNet-MoE path (BASELINE config 5): each new C-ABI kernel against plain torch fp32 on the CPU,
and the whole backbone (forward, routing, gate loss, every parameter gradient, BatchNorm running statistics) against the
reference-generated goldens / the CPU oracle.  Tolerance: 1e-3 max-norm relative (north-star), router indices exact."""
import glob
import os

import pytest
import torch
import torch.nn.functional as F

from oracle.cases import LSK_CASES, lsk_injections, upstream_grads
from oracle.lsk_moe_oracle import LskConfig, lsk_backbone_forward, lsk_param_shapes
from sm3det_b200.synth import make_images, make_state_dict
from parity_util import GAP_TOL, MAX_FLIP_FRACTION, assert_flips_are_near_ties, flipped_tokens
from sm3det_b200 import lsk_functional as LF

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), 'golden')
TOL = 1e-3


def rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-30)).item()


@pytest.fixture(scope='module')
def ops():
    from sm3det_b200 import ops as o
    return o


@pytest.mark.parametrize('ks,dil', [(3, 1), (5, 1), (7, 3)])
@pytest.mark.parametrize('C,H,W', [(32, 8, 8), (64, 19, 33), (128, 16, 16), (64, 64, 64), (32, 50, 70), (64, 96, 96)])
def test_dwconv_generic(ops, ks, dil, C, H, W):
    g = torch.Generator().manual_seed(C + H + ks)
    N = 1 if H in (50, 64) else 2    # the 256^2 .. 1024^2 levels of config 5 are multi-tile in both directions
    x = torch.randn(N, C, H, W, generator=g, requires_grad=True)
    w = (torch.randn(C, 1, ks, ks, generator=g) * 0.2).requires_grad_(True)
    b = (torch.randn(C, generator=g) * 0.1).requires_grad_(True)
    y = F.conv2d(x, w, b, padding=dil * (ks // 2), dilation=dil, groups=C)
    dy = torch.randn(y.shape, generator=g)
    y.backward(dy)
    xd = x.detach().permute(0, 2, 3, 1).contiguous().cuda()
    wt = w.detach().reshape(C, -1).t().contiguous().cuda()
    yd = ops.dwconv(xd, wt, b.detach().cuda(), ks=ks, dil=dil)
    assert rel(yd.permute(0, 3, 1, 2), y) < 1e-5
    dyd = dy.permute(0, 2, 3, 1).contiguous().cuda()
    wf = w.detach().flip(2, 3).reshape(C, -1).t().contiguous().cuda()
    dxd = ops.dwconv(dyd, wf, None, ks=ks, dil=dil)
    assert rel(dxd.permute(0, 3, 1, 2), x.grad) < 1e-5
    dwt = torch.zeros(ks * ks, C, device='cuda'); db = torch.zeros(C, device='cuda')
    ops.dwconv_wgrad(xd, dyd, dwt, db, ks=ks, dil=dil)
    assert rel(dwt.t().reshape(C, 1, ks, ks), w.grad) < 2e-5 and rel(db, b.grad) < 2e-5


@pytest.mark.parametrize('C,rows', [(64, 1000), (320, 77), (2048, 513)])
def test_colstat_affine_batchnorm(ops, C, rows):
    from sm3det_b200.lsk_functional import BatchNormFn
    g = torch.Generator().manual_seed(C)
    x = (torch.randn(rows, C, generator=g) * 1.7 + 0.6)
    w = torch.rand(C, generator=g) + 0.5; b = torch.randn(C, generator=g) * 0.1
    rm = torch.randn(C, generator=g) * 0.1; rv = torch.rand(C, generator=g) + 0.5
    dy = torch.randn(rows, C, generator=g)
    for train in (True, False):
        xr = x.clone().requires_grad_(True); wr = w.clone().requires_grad_(True); br = b.clone().requires_grad_(True)
        rm_c, rv_c = rm.clone(), rv.clone()
        ref = F.batch_norm(xr.t().reshape(1, C, rows), rm_c, rv_c, wr, br, train, 0.1, 1e-5).reshape(C, rows).t()
        ref.backward(dy)
        xg = x.cuda().requires_grad_(True); wg = w.cuda().requires_grad_(True); bg = b.cuda().requires_grad_(True)
        rm_g, rv_g = rm.cuda(), rv.cuda()
        y = BatchNormFn.apply(xg.view(1, 1, rows, C), wg, bg, rm_g, rv_g, train, 0.1, 1e-5, False)
        y.backward(dy.cuda().view(1, 1, rows, C))
        assert rel(y.view(rows, C), ref) < 2e-5
        assert rel(xg.grad, xr.grad) < 5e-5 and rel(wg.grad, wr.grad) < 5e-5 and rel(bg.grad, br.grad) < 5e-5
        assert rel(rm_g, rm_c) < 1e-5 and rel(rv_g, rv_c) < 1e-5
    s1, s2 = ops.colstat(x.cuda(), rows=rows, Cc=C)
    assert rel(s1, x.sum(0)) < 1e-5 and rel(s2, (x * x).sum(0)) < 1e-5
    out = ops.affine(x.cuda(), a1=w.cuda(), x2=dy.cuda(), a2=b.cuda(), b=rm.cuda(), add=x.cuda())
    assert rel(out, x * w + dy * b + rm + x) < 1e-6


@pytest.mark.parametrize('Ch,H,W', [(32, 8, 8), (64, 13, 21), (160, 16, 16), (32, 64, 64), (64, 40, 56), (64, 96, 96), (32, 192, 192)])
def test_lsk_select(ops, Ch, H, W):
    from sm3det_b200.lsk_functional import LSKSelectFn
    g = torch.Generator().manual_seed(Ch + H)
    N = 1 if H in (40, 64) else 2
    a1 = torch.randn(N, Ch, H, W, generator=g, requires_grad=True)
    a2 = torch.randn(N, Ch, H, W, generator=g, requires_grad=True)
    wsq = (torch.randn(2, 2, 7, 7, generator=g) * 0.2).requires_grad_(True)
    bsq = (torch.randn(2, generator=g) * 0.1).requires_grad_(True)
    attn = torch.cat([a1, a2], 1)
    agg = torch.cat([attn.mean(1, keepdim=True), attn.max(1, keepdim=True)[0]], 1)
    sig = F.conv2d(agg, wsq, bsq, padding=3).sigmoid()
    ref = a1 * sig[:, 0:1] + a2 * sig[:, 1:2]
    d = torch.randn(ref.shape, generator=g)
    ref.backward(d)
    nhwc = lambda t: t.detach().permute(0, 2, 3, 1).contiguous().cuda()
    a1g, a2g = nhwc(a1).requires_grad_(True), nhwc(a2).requires_grad_(True)
    wg, bg = wsq.detach().cuda().requires_grad_(True), bsq.detach().cuda().requires_grad_(True)
    out = LSKSelectFn.apply(a1g, a2g, wg, bg)
    out.backward(nhwc(d))
    assert rel(out.permute(0, 3, 1, 2), ref) < 1e-5
    assert rel(a1g.grad.permute(0, 3, 1, 2), a1.grad) < 2e-5 and rel(a2g.grad.permute(0, 3, 1, 2), a2.grad) < 2e-5
    assert rel(wg.grad, wsq.grad) < 5e-5 and rel(bg.grad, bsq.grad) < 5e-5


@pytest.mark.parametrize('N,H,W', [(2, 32, 48), (1, 128, 96)])
@pytest.mark.parametrize('Ci,Co,ks,stride,nchw', [(3, 64, 7, 4, True), (64, 128, 3, 2, False), (128, 320, 3, 2, False), (64, 64, 3, 2, True)])
def test_patch_embed(ops, Ci, Co, ks, stride, nchw, N, H, W):
    from sm3det_b200.lsk_functional import PatchEmbedFn
    g = torch.Generator().manual_seed(Ci + Co)
    x = torch.randn(N, Ci, H, W, generator=g, requires_grad=True)
    w = (torch.randn(Co, Ci, ks, ks, generator=g) / (Ci * ks * ks) ** 0.5).requires_grad_(True)
    b = (torch.randn(Co, generator=g) * 0.1).requires_grad_(True)
    ref = F.conv2d(x, w, b, stride=stride, padding=ks // 2)
    d = torch.randn(ref.shape, generator=g)
    ref.backward(d)
    xin = (x.detach().cuda() if nchw else x.detach().permute(0, 2, 3, 1).contiguous().cuda()).requires_grad_(Ci != 3)
    wg, bg = w.detach().cuda().requires_grad_(True), b.detach().cuda().requires_grad_(True)
    y = PatchEmbedFn.apply(xin, wg, bg, stride, nchw)
    y.backward(d.permute(0, 2, 3, 1).contiguous().cuda())
    assert rel(y.permute(0, 3, 1, 2), ref) < 5e-5
    assert rel(wg.grad, w.grad) < 1e-4 and rel(bg.grad, b.grad) < 1e-4
    if Ci != 3:
        assert rel(xin.grad if nchw else xin.grad.permute(0, 3, 1, 2), x.grad) < 1e-4


def test_linear_gelu_mul_axpy(ops):
    from sm3det_b200.lsk_functional import AxpyFn, GeluFn, LinearFn, MulFn
    g = torch.Generator().manual_seed(3)
    T, K, N = 300, 64, 160
    x = torch.randn(T, K, generator=g, requires_grad=True)
    w = (torch.randn(N, K, 1, 1, generator=g) / 8).requires_grad_(True)
    b = (torch.randn(N, generator=g) * 0.1).requires_grad_(True)
    ls = (torch.rand(N, generator=g) + 0.1).requires_grad_(True)
    sc = torch.randn(T, N, generator=g, requires_grad=True)
    rs = (torch.rand(T, generator=g) > 0.3).float() / 0.7
    h = F.gelu(F.linear(x, w.view(N, K), b))
    ref = sc + rs[:, None] * ls * (F.gelu(h) * sc)
    d = torch.randn(T, N, generator=g)
    ref.backward(d)
    xg, wg, bg, lg, sg = (t.detach().cuda().requires_grad_(True) for t in (x, w, b, ls, sc))
    hg = LinearFn.apply(xg, wg, bg, True)
    out = AxpyFn.apply(MulFn.apply(GeluFn.apply(hg), sg), sg, lg, rs.cuda())
    out.backward(d.cuda())
    assert rel(out, ref) < 5e-5
    for a, r, name in ((xg, x, 'x'), (wg, w, 'w'), (bg, b, 'b'), (lg, ls, 'ls'), (sg, sc, 'sc')):
        assert rel(a.grad, r.grad) < 2e-4, name


# ------------------------------------------------------------------------------------------------
def build(kw, seed=0, unit='lsk'):
    from sm3det_b200 import LSKNet_moe_MultiInput, VAN_moe_MultiInput
    cfg = LskConfig(spatial_unit=unit, **kw)
    sd = make_state_dict(lsk_param_shapes(cfg), seed, True)
    net = (LSKNet_moe_MultiInput if unit == 'lsk' else VAN_moe_MultiInput)(norm_cfg=dict(type='SyncBN', requires_grad=True), **kw)
    net.load_state_dict(sd, strict=True)
    return cfg, sd, net.cuda()


def inject(net, cfg, noise, drops):
    ni = iter(noise or [])
    di = iter(drops or [])
    for i in range(cfg.num_stages):
        for blk in getattr(net, f'block{i + 1}'):
            for fc in (blk.mlp.fc1, blk.mlp.fc2):
                if hasattr(fc, 'experts') and noise is not None:
                    fc._injected_noise = next(ni)
            if drops is not None:
                m1, m2 = next(di), next(di)
                blk.mlp._injected_drop_masks = [m1.permute(0, 2, 3, 1).contiguous(), m2.permute(0, 2, 3, 1).contiguous()]


@pytest.mark.parametrize('path', sorted(glob.glob(os.path.join(GOLD, 'lsk_*.pt')) + glob.glob(os.path.join(GOLD, 'van_*.pt'))), ids=lambda p: os.path.basename(p)[:-3])
def test_lsk_backbone_matches_reference_golden(path):
    gold = torch.load(path, weights_only=False)
    cfg, sd, net = build(gold['kw'], unit=gold.get('unit', 'lsk'))
    n, h, w = gold['img']
    x = make_images(n, h, w, seed=1234).cuda()
    train = gold['mode'] != 'eval'
    net.train(train)
    noise, drops = lsk_injections(cfg, gold)
    inject(net, cfg, noise, drops)
    rec, amax = [], []
    LF.AMAX_RECORD = amax
    try:
        with torch.set_grad_enabled(train):
            res = net(x, record=rec)
    finally:
        LF.AMAX_RECORD = None
    has_loss = 'gate_loss' in gold
    outs, loss = res if has_loss else (res, None)
    st = gold.get('stride', 1)
    full = bool(gold['moe']) and 'gap' in gold['moe'][0]
    flips = sum(int(flipped_tokens(r['top_idx'], g['top_idx']).sum()) for r, g in zip(rec, gold['moe']))
    if not full:
        assert flips == 0, 'router indices must be bit-exact on the small fixtures'
    ups = upstream_grads([o.detach().cpu() for o in outs])
    if train:
        (sum((o * g.cuda()).sum() for o, g in zip(outs, ups)) + (loss if has_loss else 0.0)).backward()
    new_sd = net.state_dict()

    def grad_tol(name):
        return 1e-2 if name.endswith('w_gate.temperature') else 3e-3     # scalar sum over all tokens with heavy cancellation

    def zero_grad_bias(name):
        # a conv bias in front of a training-mode BatchNorm: the true gradient is exactly 0, both sides hold fp32 noise
        return name.endswith('proj.bias') or name == 'dataset_stems.single.bias'

    # LSKblock's channel max (lsk_moe.py:337) is the second discrete selection on this path: at 10^4..10^5 tokens per level a few
    # tokens have their two largest channels closer than the 3e-5 forward error, and ONE flipped token moves the whole d(max) of
    # that token (a 7x7x2-tap sum over all channels) to another channel -- percent-level changes in the conv1/conv2 gradients
    # (profiles/r02_lsk_argmax_flips.txt).  The forced-oracle pass below follows the CUDA path's channel choice, counts the
    # tokens where that differs from the oracle's own argmax and requires each of them to be a numerical tie.
    amax_flips, arec = 0, []
    is_lsk = gold.get('unit', 'lsk') == 'lsk'
    if full or flips > 0:
        # ---- the oracle teacher-forced to the CUDA path's routing: every element, every gradient (tests/parity_util.py) ----
        forced = [r['top_idx'].cpu().long() for r in rec]
        sdo = {k: (v.clone().requires_grad_(True) if train and v.is_floating_point() and not any(t in k for t in ('running_', 'num_batches', '.mean', '.std')) else v)
               for k, v in sd.items()}
        bn_state = {}
        rec_c = []
        with torch.set_grad_enabled(train):
            res_c = lsk_backbone_forward(sdo, cfg, x.cpu(), train=train, noise=noise, drop_masks=drops, bn_state=bn_state, forced_idx=forced,
                                         record=rec_c, forced_amax=[a.cpu() for a in amax] if is_lsk else None, amax_record=arec)
        oc, lc = res_c if has_loss else (res_c, None)
        for a in arec:
            flip = a['own'] != a['forced']
            amax_flips += int(flip.sum())
            if flip.any():
                assert float((a['gap'][flip] / a['scale'][flip]).max()) < GAP_TOL, (a['prefix'], 'channel-argmax flip is not a near-tie')
            assert int(flip.sum()) <= max(2, MAX_FLIP_FRACTION * flip.numel()), (a['prefix'], int(flip.sum()), flip.numel())
        print(os.path.basename(path), 'channel-argmax flips', amax_flips, 'of', sum(a['own'].numel() for a in arec))
        # per layer: the CUDA routing vs the oracle's own top-k on the same (forced-upstream) inputs -- numerical ties only
        own = [dict(top_idx=c['logits'].topk(g['top_idx'].shape[1], dim=-1).indices, logits=c['logits']) for g, c in zip(rec, rec_c)]
        own_flips = assert_flips_are_near_ties(rec, own, what=gold['name'])
        assert own_flips > 0 or flips == 0, 'routing differs from the fixture although every layer agrees with the oracle'
        errs = [rel(a, b) for a, b in zip(outs, oc)]
        print(os.path.basename(path), 'flips', flips, 'rel errs vs forced oracle', errs)
        assert max(errs) < TOL
        if has_loss:
            assert abs(loss.item() - lc.item()) <= 1e-4 * abs(lc.item()) + 1e-8
        if train:
            (sum((o * g).sum() for o, g in zip(oc, ups)) + (lc if has_loss else 0.0)).backward()
            bad = []
            for name, p in net.named_parameters():
                want = sdo[name].grad
                if want is None:
                    want = torch.zeros_like(sdo[name])
                got = p.grad.detach().float().cpu()
                if zero_grad_bias(name):
                    assert (got - want).abs().max().item() < 1e-5, name
                    continue
                e = ((got - want).abs().max() / max(want.abs().max().item(), 1e-5)).item()
                bad.append((e / grad_tol(name), e, name))
            bad.sort(reverse=True)
            print('worst grads vs forced oracle', bad[:5])
            assert bad[0][0] < 1.0, bad[:8]
            for k, v in bn_state.items():
                assert rel(new_sd[k], v) < 1e-4, k
    if flips == 0:
        # ---- the reference-generated fixture itself ----
        errs = [rel(o[:, :, ::st, ::st], g) for o, g in zip(outs, gold['outs'])]
        print(os.path.basename(path), 'rel errs vs fixture', errs)
        assert max(errs) < TOL
        if has_loss:
            assert abs(loss.item() - gold['gate_loss'].item()) <= 1e-4 * abs(gold['gate_loss'].item()) + 1e-8
        if train and amax_flips == 0:
            bad = []
            for name, p in net.named_parameters():
                gg = gold['grads'].get(name)
                if gg is None:
                    continue
                got = p.grad.detach().float().cpu().reshape(-1)
                if 'full' in gg:
                    want = gg['full']
                else:
                    want, got = gg['sample'], got[gg['idx']]
                scale = (gg['l2'] / (p.numel() ** 0.5)) if 'l2' in gg else want.abs().max().item()
                if zero_grad_bias(name):
                    assert (got - want).abs().max().item() < 1e-5, name
                    continue
                e = ((got - want).abs().max() / max(want.abs().max().item(), scale, 1e-5)).item()
                bad.append((e / grad_tol(name), e, name))
            bad.sort(reverse=True)
            print('worst grads vs fixture', bad[:14])
            assert bad[0][0] < 1.0, bad[:8]
            for k, v in gold['bn'].items():
                assert rel(new_sd[k], v) < 1e-4, k


def test_lsk_eval_list_input_and_plain_class():
    """list input is concatenated on the batch (lsk_moe.py:751-754); LSKNet_moe (plain) returns the same maps."""
    spec = LSK_CASES['lsk_mini_moe_e4k2_eval']
    cfg, sd, net = build(spec['kw'])
    net.eval()
    x = make_images(2, 64, 64, seed=9)
    with torch.no_grad():
        o1, l1 = net(x.cuda())
        o2, l2 = net([x[:1].cuda(), x[1:].cuda()], datasets=['a', 'b'])
        ref, rl = lsk_backbone_forward(sd, cfg, x, train=False)
    assert all(torch.equal(a, b) for a, b in zip(o1, o2))
    assert max(rel(a, b) for a, b in zip(o1, ref)) < TOL and abs(l1.item() - rl.item()) < 1e-4 * abs(rl.item())
    assert all(o.is_contiguous() and o.shape[0] == 2 for o in o1)


def test_fused_dropout(ops):
    """sm3_dropout: keep-rate ~ 1-p, survivors scaled by 1/(1-p), the backward reuses the identical mask, seeds differ."""
    from sm3det_b200.lsk_functional import DropoutFn
    # seeded, and free of exact zeros (which would read as dropped below)
    x = torch.randn(1 << 20, generator=torch.Generator().manual_seed(0)).cuda().requires_grad_(True)
    assert bool((x != 0).all())
    y = DropoutFn.apply(x, 0.1, 1234)
    keep = (y != 0)
    assert abs(keep.float().mean().item() - 0.9) < 3e-3
    assert torch.allclose(y[keep], x.detach()[keep] / 0.9)
    y.backward(torch.ones_like(y))
    assert torch.equal(x.grad != 0, keep) and torch.allclose(x.grad[keep], torch.full_like(x.grad[keep], 1 / 0.9))
    y2 = ops.dropout(x.detach(), 0.1, 1235)
    assert (y2 != 0).ne(keep).float().mean().item() > 0.1            # a different seed gives a different mask
    assert torch.equal(ops.dropout(x.detach(), 0.0, 7), x.detach())


@pytest.mark.parametrize('C,Co,H', [(64, 128, 8), (128, 128, 4), (64, 64, 16), (128, 128, 16)])
@pytest.mark.parametrize('N', [2, 1])
def test_stage_boundary_norm_output_feeds_next_patch_embed(ops, N, C, Co, H):
    """lsk_moe.py:551-559: the per-stage LayerNorm output (NCHW) is BOTH a returned feature (its own loss term) and the
    input of the next OverlapPatchEmbed (3x3/s2 conv + BatchNorm): two gradient contributions meet at one tensor.
    Found at the real config-5 shapes (batch 1 per image): checked here for N = 1 and N = 2."""
    from sm3det_b200 import functional as Fn
    from sm3det_b200.lsk_functional import BatchNormFn, PatchEmbedFn
    g = torch.Generator().manual_seed(5 + N)
    W = H
    x = torch.randn(N, H, W, C, generator=g, requires_grad=True)
    lw = (torch.rand(C, generator=g) + 0.5).requires_grad_(True); lb = (torch.randn(C, generator=g) * 0.1).requires_grad_(True)
    cw = (torch.randn(Co, C, 3, 3, generator=g) / (9 * C) ** 0.5).requires_grad_(True); cb = (torch.randn(Co, generator=g) * 0.1).requires_grad_(True)
    bw = (torch.rand(Co, generator=g) + 0.5).requires_grad_(True); bb = (torch.randn(Co, generator=g) * 0.1).requires_grad_(True)
    rm, rv = torch.randn(Co, generator=g) * 0.1, torch.rand(Co, generator=g) + 0.5
    g1 = torch.randn(N, C, H, W, generator=g); g2 = torch.randn(N, Co, H // 2, W // 2, generator=g)
    # torch reference
    y = F.layer_norm(x, (C,), lw, lb, 1e-6).permute(0, 3, 1, 2).contiguous()
    z = F.batch_norm(F.conv2d(y, cw, cb, stride=2, padding=1), rm.clone(), rv.clone(), bw, bb, True, 0.1, 1e-5)
    ((y * g1).sum() + (z * g2).sum()).backward()
    # CUDA path
    d = lambda t: t.detach().cuda().requires_grad_(True)
    xg, lwg, lbg, cwg, cbg, bwg, bbg = d(x), d(lw), d(lb), d(cw), d(cb), d(bw), d(bb)
    yg = Fn.OutNormFn.apply(xg, lwg, lbg, 1e-6)
    zg = BatchNormFn.apply(PatchEmbedFn.apply(yg, cwg, cbg, 2, True), bwg, bbg, rm.cuda(), rv.cuda(), True, 0.1, 1e-5, False)
    ((yg * g1.cuda()).sum() + (zg * g2.permute(0, 2, 3, 1).contiguous().cuda()).sum()).backward()
    assert rel(yg, y) < 2e-5 and rel(zg.permute(0, 3, 1, 2), z) < (5e-5 if N * H * W >= 64 else 3e-4)   # BN over 4 tokens amplifies rounding
    for a, r, name in ((xg, x, 'x'), (lwg, lw, 'ln.w'), (lbg, lb, 'ln.b'), (cwg, cw, 'conv.w'), (bwg, bw, 'bn.w'), (bbg, bb, 'bn.b')):
        assert rel(a.grad, r.grad) < 3e-4, (name, rel(a.grad, r.grad))
