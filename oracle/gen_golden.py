"""Generate tests/golden/*.pt by running the UNMODIFIED reference (via oracle/ref_shim.py).

Run in the build container only (needs /root/reference):  python -m oracle.gen_golden
Every case also asserts that the restated oracle reproduces the reference bit-for-bit on CPU
(forward outputs, gate loss, routing decisions, parameter gradients) -- this is what pins the
oracle.  Fixtures hold no weights: those are regenerated from seeds by sm3det_b200.synth.
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_shim                                   # noqa: E402
from oracle.cases import CASES, make_noise, summarize_grad, upstream_grads   # noqa: E402
from oracle.convnext_moe_oracle import OracleConfig, backbone_forward, param_shapes, tie_da_weights  # noqa: E402
from sm3det_b200.synth import make_images, make_state_dict, state_dict_checksum    # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')


def moe_token_counts(cfg, n, h, w):
    counts = []
    for i in range(4):
        t = n * (h // (4 * 2 ** i)) * (w // (4 * 2 ** i))
        counts += [t] * len(cfg.moe_blocks(i))
    return counts


def moe_digest(r, full):
    """What a fixture keeps of one MoE layer.  Full-size cases: int8 indices + the (k)-vs-(k+1) logit gap per token (the
    margin a routing flip is judged against) instead of the gate values."""
    d = dict(prefix=r['prefix'], importance=r['importance'], load=r['load'], loss=r['loss'])
    if not full:
        d.update(top_idx=r['top_idx'].to(torch.int16), top_gates=r['top_gates'])
        return d
    k = r['top_idx'].shape[1]
    lg = r['logits']
    top = lg.topk(min(k + 1, lg.shape[1]), dim=-1).values
    d.update(top_idx=r['top_idx'].to(torch.int8), logit_scale=float(lg.abs().max()),
             gap=(top[:, k - 1] - top[:, k]).float() if top.shape[1] > k else torch.full((lg.shape[0],), float('inf')))
    return d


def run_case(name, spec):
    kw = dict(spec['kw'])
    da = bool(spec.get('da', False))
    datasets = spec.get('datasets')
    cfg = OracleConfig(da=da, **kw)
    if da:
        net = ref_shim.build_reference_backbone('ConvNeXt_DA_MultiInput', seed=0, module='convnext_moe_DA', **kw)
    else:
        net = ref_shim.build_reference_backbone('ConvNeXt_moe_MultiInput', seed=0, **kw)
    call = (lambda inp: net(inp, datasets)) if da else net
    okw = dict(datasets=datasets) if da else {}
    shapes = param_shapes(cfg)
    rsd = net.state_dict()
    assert set(shapes) == set(rsd), set(shapes) ^ set(rsd)
    for k, s in shapes.items():
        assert tuple(rsd[k].shape) == tuple(s), k
    sd = make_state_dict(shapes, seed=0, trained_like=(spec['weights'] == 'trained'))
    if da:
        tie_da_weights(sd)                      # the reference registers ONE Sequential three times (fc.2's values survive a load)
    net.load_state_dict(sd, strict=True)
    n, h, w = spec['img']
    x = make_images(n, h, w, seed=1234)
    mode = spec['mode']
    gold = dict(name=name, kw=kw, img=spec['img'], mode=mode, weights=spec['weights'],
                sd_checksum=state_dict_checksum(sd), x_checksum=float(x.double().abs().sum()))
    if da:
        gold.update(da=True, datasets=list(datasets))
        if len(datasets) > 1:
            x = [x[i:i + 1] for i in range(n)]      # the detector passes one tensor per modality (trisource detector :141-153)
    record = []
    st = spec['stride']
    if mode == 'eval':
        net.eval()
        with torch.no_grad():
            ref = call(x)
            orc = backbone_forward(sd, cfg, x, train=False, record=record, **okw)
    else:
        net.train()
        noise = None
        if mode == 'train_noisy':
            noise = make_noise(cfg, moe_token_counts(cfg, n, h, w))
            it = iter(noise)
            orig = torch.randn_like
            torch.randn_like = lambda t, *a, **k: next(it).to(t.dtype)   # inject the noise stream
        try:
            ref = call(x)
        finally:
            if mode == 'train_noisy':
                torch.randn_like = orig
        sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and 'ffn.mean' not in k and 'ffn.std' not in k else v)
               for k, v in sd.items()}
        if da:
            tie_da_weights(sdg)
        orc = backbone_forward(sdg, cfg, x, train=True, noise=noise, record=record, **okw)
    has_loss = isinstance(ref, tuple) and len(ref) == 2 and isinstance(ref[0], tuple)
    r_outs, r_loss = (ref if has_loss else (ref, None))
    o_outs, o_loss = (orc if has_loss else (orc, None))
    for a, b in zip(r_outs, o_outs):
        assert torch.equal(a, b), f'{name}: oracle output differs from reference by {(a - b).abs().max()}'
    if has_loss:
        assert torch.equal(r_loss, o_loss), (r_loss, o_loss)
        gold['gate_loss'] = r_loss.detach().clone()
    gold['outs'] = [o.detach()[:, :, ::st, ::st].clone() for o in r_outs]
    gold['out_l2'] = [o.detach().double().norm().item() for o in r_outs]
    gold['stride'] = st
    gold['moe'] = [moe_digest(r, spec.get('full', False)) for r in record]
    if mode != 'eval':
        ups = upstream_grads(r_outs)
        (sum((o * g).sum() for o, g in zip(r_outs, ups)) + (r_loss if has_loss else 0.0)).backward()
        (sum((o * g).sum() for o, g in zip(o_outs, ups)) + (o_loss if has_loss else 0.0)).backward()
        grads = {}
        for pname, p in net.named_parameters():
            og = sdg[pname].grad
            if p.grad is None:
                assert og is None or float(og.abs().max()) == 0.0, pname
                continue
            assert og is not None, pname
            if spec.get('full', False):
                # multi-threaded CPU reductions over >= 10^5 tokens are not run-to-run bit-stable (the reference differs
                # from ITSELF in the last bit between runs); forward outputs, loss and routing above stay bit-exact
                assert float((p.grad - og).abs().max()) <= 1e-5 * float(og.abs().max()) + 1e-12, \
                    f'{name}: grad {pname} differs by {(p.grad - og).abs().max()}'
            else:
                assert torch.equal(p.grad, og), f'{name}: grad {pname} differs by {(p.grad - og).abs().max()}'
            # thousands of expert parameters (config 4): keep the digests small -- the GPU test compares full gradients
            # against the live oracle anyway, the digests only pin oracle == reference
            grads[pname] = summarize_grad(p.grad, 256, 24) if len(shapes) > 1500 else summarize_grad(p.grad)
        gold['grads'] = grads
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + '.pt')
    torch.save(gold, path)
    print(f'{name}: ok, {os.path.getsize(path) / 1024:.0f} KiB, moe layers {len(record)}')


def run_lsk_case(name, spec):
    """LSKNet-MoE: run the unmodified reference lsk_moe.py, assert the restated oracle reproduces it bit-for-bit
    (outputs, gate loss, routing, parameter gradients, BatchNorm running statistics), save the fixture."""
    import torch.nn.functional as F
    from oracle.cases import lsk_plan, make_drop_masks
    from oracle.lsk_moe_oracle import LskConfig, lsk_backbone_forward, lsk_param_shapes
    kw = dict(spec['kw'])
    unit = spec.get('unit', 'lsk')
    cfg = LskConfig(spatial_unit=unit, **kw)
    mod = ref_shim.load_reference_module('lsk_moe' if unit == 'lsk' else 'van_moe')
    torch.manual_seed(0)
    cls = mod.LSKNet_moe_MultiInput if unit == 'lsk' else mod.VAN_moe_MultiInput
    net = cls(norm_cfg=dict(type='SyncBN', requires_grad=True), **kw)
    shapes = lsk_param_shapes(cfg)
    rsd = net.state_dict()
    assert set(shapes) == set(rsd), set(shapes) ^ set(rsd)
    for k, sh in shapes.items():
        assert tuple(rsd[k].shape) == tuple(sh), k
    sd = make_state_dict(shapes, seed=0, trained_like=True)
    net.load_state_dict(sd, strict=True)
    n, h, w = spec['img']
    x = make_images(n, h, w, seed=1234)
    mode = spec['mode']
    gold = dict(name=name, kw=kw, img=spec['img'], mode=mode, weights='trained', family='lsk', unit=unit,
                sd_checksum=state_dict_checksum({k: v.float() for k, v in sd.items()}), x_checksum=float(x.double().abs().sum()))
    record, bn_state = [], {}
    no_grad_keys = ('running_', 'num_batches', '.mean', '.std')
    if mode == 'eval':
        net.eval()
        with torch.no_grad():
            ref = net(x)
            orc = lsk_backbone_forward(sd, cfg, x, train=False, record=record)
    else:
        net.train()
        noise = drops = None
        tokens, dshapes = lsk_plan(cfg, n, h, w)
        orig_randn, orig_drop = torch.randn_like, F.dropout
        if mode == 'train_noisy':
            noise = [torch.randn(t, cfg.num_experts, generator=torch.Generator().manual_seed(7 + i)) for i, t in enumerate(tokens)]
            it = iter(noise)
            torch.randn_like = lambda t, *a, **k: next(it).to(t.dtype)
        if cfg.drop_rate > 0:
            drops = make_drop_masks(dshapes, cfg.drop_rate)
            dit = iter(drops)
            F.dropout = lambda t, p=0.5, training=True, inplace=False: t * next(dit) if training else t
        try:
            ref = net(x)
        finally:
            torch.randn_like, F.dropout = orig_randn, orig_drop
        sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and not any(t in k for t in no_grad_keys) else v)
               for k, v in sd.items()}
        orc = lsk_backbone_forward(sdg, cfg, x, train=True, noise=noise, drop_masks=drops, record=record, bn_state=bn_state)
    has_loss = isinstance(ref, tuple) and len(ref) == 2 and isinstance(ref[0], tuple)
    r_outs, r_loss = (ref if has_loss else (ref, None))
    o_outs, o_loss = (orc if has_loss else (orc, None))
    for a, b in zip(r_outs, o_outs):
        assert torch.equal(a, b), f'{name}: oracle output differs from reference by {(a - b).abs().max()}'
    if has_loss:
        assert torch.equal(r_loss, o_loss), (r_loss, o_loss)
        gold['gate_loss'] = r_loss.detach().clone()
    st = spec.get('stride', 1)
    gold['outs'] = [o.detach()[:, :, ::st, ::st].clone() for o in r_outs]
    gold['out_l2'] = [o.detach().double().norm().item() for o in r_outs]
    gold['stride'] = st
    gold['moe'] = [moe_digest(r, spec.get('full', False)) for r in record]
    if mode != 'eval':
        ups = upstream_grads(r_outs)
        (sum((o * g).sum() for o, g in zip(r_outs, ups)) + (r_loss if has_loss else 0.0)).backward()
        (sum((o * g).sum() for o, g in zip(o_outs, ups)) + (o_loss if has_loss else 0.0)).backward()
        grads = {}
        for pname, p in net.named_parameters():
            og = sdg[pname].grad
            if p.grad is None:
                assert og is None or float(og.abs().max()) == 0.0, pname
                continue
            assert og is not None, pname
            if spec.get('full', False):
                # multi-threaded CPU reductions over >= 10^5 tokens are not run-to-run bit-stable (the reference differs
                # from ITSELF in the last bit between runs); forward outputs, loss and routing above stay bit-exact
                assert float((p.grad - og).abs().max()) <= 1e-5 * float(og.abs().max()) + 1e-12, \
                    f'{name}: grad {pname} differs by {(p.grad - og).abs().max()}'
            else:
                assert torch.equal(p.grad, og), f'{name}: grad {pname} differs by {(p.grad - og).abs().max()}'
            grads[pname] = summarize_grad(p.grad)
        gold['grads'] = grads
        new_sd = net.state_dict()
        for k, v in bn_state.items():
            assert torch.equal(v, new_sd[k]), k
        gold['bn'] = {k: v.clone() for k, v in bn_state.items()}
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + '.pt')
    torch.save(gold, path)
    print(f'{name}: ok, {os.path.getsize(path) / 1024:.0f} KiB, moe layers {len(record)}')


if __name__ == '__main__':
    from oracle.cases import GOLDEN_THREADS, LSK_CASES
    torch.set_num_threads(GOLDEN_THREADS)
    names = sys.argv[1:] or (list(CASES) + list(LSK_CASES))
    for nm in names:
        if nm in LSK_CASES:
            run_lsk_case(nm, LSK_CASES[nm])
        else:
            run_case(nm, CASES[nm])
