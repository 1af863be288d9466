"""The CPU oracle against (a) the committed golden fixtures generated from the unmodified reference
and (b) the reference modules' own outputs recorded by oracle/gen_reference_snapshots.py."""
import glob
import os

import pytest
import torch

from oracle import gen_reference_snapshots
from oracle.cases import CASES, assert_matches_summary, golden_threads, make_noise, summarize_grad, upstream_grads
from oracle.convnext_moe_oracle import OracleConfig, backbone_forward, param_shapes, tie_da_weights
from oracle.gen_golden import moe_token_counts
from sm3det_b200.synth import make_images, make_state_dict, state_dict_checksum

GOLD = os.path.join(os.path.dirname(__file__), 'golden')


@pytest.fixture(autouse=True)
def _golden_threads():
    with golden_threads():
        yield


def _run_oracle(gold, record):
    kw = gold['kw']
    da = bool(gold.get('da'))
    cfg = OracleConfig(da=da, **kw)
    sd = make_state_dict(param_shapes(cfg), 0, gold['weights'] == 'trained')
    okw = {}
    if da:
        tie_da_weights(sd)
        okw = dict(datasets=gold['datasets'])
    assert abs(state_dict_checksum(sd) - gold['sd_checksum']) <= 1e-9 * abs(gold['sd_checksum']), 'weight RNG drift'
    n, h, w = gold['img']
    x = make_images(n, h, w, seed=1234)
    assert abs(float(x.double().abs().sum()) - gold['x_checksum']) <= 1e-9 * gold['x_checksum'], 'image RNG drift'
    mode = gold['mode']
    if da and len(gold['datasets']) > 1:
        x = [x[i:i + 1] for i in range(n)]
    if mode == 'eval':
        with torch.no_grad():
            return cfg, sd, backbone_forward(sd, cfg, x, train=False, record=record, **okw)
    noise = make_noise(cfg, moe_token_counts(cfg, n, h, w)) if mode == 'train_noisy' else None
    sdg = {k: (v.clone().requires_grad_(True) if 'ffn.mean' not in k and 'ffn.std' not in k else v) for k, v in sd.items()}
    if da:
        tie_da_weights(sdg)
    return cfg, sdg, backbone_forward(sdg, cfg, x, train=True, noise=noise, record=record, **okw)


@pytest.mark.parametrize('path', sorted(p for p in glob.glob(os.path.join(GOLD, '*.pt')) if not os.path.basename(p).startswith(('lsk_', 'van_'))), ids=lambda p: os.path.basename(p)[:-3])
def test_oracle_matches_reference_golden(path):
    gold = torch.load(path, weights_only=False)
    if gold['mode'] != 'eval' and gold['img'][1] >= 512 and not os.environ.get('SM3_SLOW_TESTS'):
        pytest.skip('full-size training fixture: re-checked by oracle/gen_golden.py (set SM3_SLOW_TESTS=1 to run here)')
    record = []
    cfg, sd, res = _run_oracle(gold, record)
    has_loss = 'gate_loss' in gold
    outs, loss = res if has_loss else (res, None)
    st = gold['stride']
    # same torch build => bit-exact; tolerate 2e-6 relative for a different CPU kernel selection
    for o, g, l2 in zip(outs, gold['outs'], gold['out_l2']):
        torch.testing.assert_close(o.detach()[:, :, ::st, ::st], g, rtol=2e-6, atol=2e-6)
        assert abs(o.detach().double().norm().item() - l2) <= 2e-6 * l2
    if has_loss:
        torch.testing.assert_close(loss.detach(), gold['gate_loss'], rtol=1e-6, atol=1e-9)
    assert len(record) == len(gold['moe'])
    for r, g in zip(record, gold['moe']):
        assert r['prefix'] == g['prefix']
        assert torch.equal(r['top_idx'].to(g['top_idx'].dtype), g['top_idx']), 'router top-k indices must be bit-exact'
        if 'top_gates' in g:
            torch.testing.assert_close(r['top_gates'], g['top_gates'], rtol=1e-6, atol=1e-7)
        torch.testing.assert_close(r['load'], g['load'], rtol=1e-6, atol=1e-6)
    if 'grads' in gold:
        ups = upstream_grads(outs)
        (sum((o * u).sum() for o, u in zip(outs, ups)) + (loss if has_loss else 0.0)).backward()
        for name, g in gold['grads'].items():
            s = summarize_grad(sd[name].grad)
            if 'full' in g:
                torch.testing.assert_close(s['full'], g['full'], rtol=1e-5, atol=1e-7)
            else:
                torch.testing.assert_close(s['sample'], g['sample'], rtol=1e-5, atol=1e-7)
                assert abs(s['l2'] - g['l2']) <= 1e-5 * (g['l2'] + 1e-12)


@pytest.mark.parametrize('name', ['mini_moe_e4k2_eval', 'mini_moe_e8k3_eval'])
def test_oracle_matches_live_reference(name):
    """Another weight seed and image than the golden fixture; the reference's outputs were recorded from the live module."""
    ref = gen_reference_snapshots.load('convnext')['live'][name]
    spec = CASES[name]
    kw = dict(spec['kw'])
    cfg = OracleConfig(**kw)
    sd = make_state_dict(param_shapes(cfg), 3, True)
    x = make_images(2, 64, 64, seed=5)
    with torch.no_grad():
        outs, loss = backbone_forward(sd, cfg, x)
    assert len(outs) == len(ref['outs'])
    for i, (o, r) in enumerate(zip(outs, ref['outs'])):
        assert_matches_summary(o, r, f'output {i}')
    assert torch.equal(loss, ref['gate_loss'])


def test_plain_convnext_moe_class_matches():
    """ConvNeXt_moe (stem inside downsample_layers.0) -- convnext_moe.py:407-600."""
    ref = gen_reference_snapshots.load('convnext')['plain']
    kw = dict(arch=dict(depths=[1, 1, 2, 1], channels=[32, 64, 96, 128]), MoE_Block_inds=[[], [], [1], []],
              num_experts=4, top_k=2)
    assert ref['kw'] == kw
    cfg = OracleConfig(multi_input=False, **kw)
    shapes = param_shapes(cfg)
    assert set(shapes) == set(ref['keys'])
    sd = make_state_dict(shapes, 1, True)
    x = make_images(1, 64, 64, seed=2)
    with torch.no_grad():
        outs = backbone_forward(sd, cfg, x)[0]
    assert len(outs) == len(ref['outs'])
    for i, (o, r) in enumerate(zip(outs, ref['outs'])):
        assert_matches_summary(o, r, f'output {i}')
