"""CPU checks for the LSKNet-MoE family: oracle vs committed goldens (generated from the real reference by
oracle/gen_golden.py), oracle vs the reference's outputs and layouts recorded by oracle/gen_reference_snapshots.py, and the
drop-in contract (state_dict keys / shapes, constructor kwargs) of the CUDA module -- no GPU compute."""
import glob
import os

import pytest
import torch

from oracle import gen_reference_snapshots
from oracle.cases import LSK_CASES, assert_matches_summary, golden_threads, lsk_injections
from oracle.lsk_moe_oracle import LskConfig, lsk_backbone_forward, lsk_param_shapes
from sm3det_b200.synth import make_images, make_state_dict

GOLD = os.path.join(os.path.dirname(__file__), 'golden')


@pytest.fixture(autouse=True)
def _golden_threads():
    with golden_threads():
        yield


def _inputs(gold):
    cfg = LskConfig(spatial_unit=gold.get('unit', 'lsk'), **gold['kw'])
    sd = make_state_dict(lsk_param_shapes(cfg), 0, True)
    n, h, w = gold['img']
    return cfg, sd, make_images(n, h, w, seed=1234)


@pytest.mark.parametrize('path', sorted(glob.glob(os.path.join(GOLD, 'lsk_*.pt')) + glob.glob(os.path.join(GOLD, 'van_*.pt'))), ids=lambda p: os.path.basename(p)[:-3])
def test_oracle_reproduces_reference_golden(path):
    gold = torch.load(path, weights_only=False)
    if gold['mode'] != 'eval' and gold['img'][1] >= 512 and not os.environ.get('SM3_SLOW_TESTS'):
        pytest.skip('full-size training fixture: re-checked by oracle/gen_golden.py (set SM3_SLOW_TESTS=1 to run here)')
    cfg, sd, x = _inputs(gold)
    assert abs(float(x.double().abs().sum()) - gold['x_checksum']) < 1e-6 * gold['x_checksum']
    noise, drops = lsk_injections(cfg, gold)
    rec, bn = [], {}
    with torch.no_grad():
        res = lsk_backbone_forward(sd, cfg, x, train=gold['mode'] != 'eval', noise=noise, drop_masks=drops, record=rec, bn_state=bn)
    outs, loss = res if 'gate_loss' in gold else (res, None)
    st = gold.get('stride', 1)
    for o, g in zip(outs, gold['outs']):
        assert torch.equal(o[:, :, ::st, ::st], g)
    if loss is not None:
        assert torch.equal(loss, gold['gate_loss'])
    for r, g in zip(rec, gold['moe']):
        assert torch.equal(r['top_idx'].to(g['top_idx'].dtype), g['top_idx'])
    for k, v in gold.get('bn', {}).items():
        assert torch.equal(bn[k], v), k


def test_oracle_matches_live_reference_lsk():
    """Another image than the golden fixture; the reference's outputs were recorded from the live module."""
    ref = gen_reference_snapshots.load('lsk')['live']
    spec = LSK_CASES['lsk_mini_moe_e4k2_eval']
    cfg = LskConfig(**spec['kw'])
    sd = make_state_dict(lsk_param_shapes(cfg), 0, True)
    x = make_images(*spec['img'], seed=5)
    with torch.no_grad():
        orc, ol = lsk_backbone_forward(sd, cfg, x, train=False)
    assert len(orc) == len(ref['outs'])
    for i, (o, r) in enumerate(zip(orc, ref['outs'])):
        assert_matches_summary(o, r, f'output {i}')
    assert torch.equal(ol, ref['gate_loss'])


def test_lsk_contract_state_dict_and_registry():
    from sm3det_b200 import LSKNet_moe, build_backbone
    kw = dict(MoE_Block_inds_fc1=[[], [0], [0, 2], [0]], MoE_Block_inds_fc2=[[], [0], [0, 2], [0]], num_experts=4, top_k=2,
              embed_dims=[64, 128, 320, 512], depths=[2, 2, 4, 2], drop_rate=0.1, drop_path_rate=0.,
              norm_cfg=dict(type='SyncBN', requires_grad=True))          # configs/SM3Det/SM3Det_lsk_s.py:13-25
    net = build_backbone(dict(type='LSKNet_moe_MultiInput', datasets=None, **kw))
    cfg = LskConfig(**{k: v for k, v in kw.items() if k != 'norm_cfg'})
    shapes = lsk_param_shapes(cfg)
    sd = net.state_dict()
    assert set(shapes) == set(sd)
    assert all(tuple(sd[k].shape) == tuple(s) for k, s in shapes.items())
    assert abs(sum(p.numel() for p in net.parameters()) / 1e6 - 27.57) < 0.01          # SURVEY Appendix B
    net.load_state_dict(make_state_dict(shapes, 0, True), strict=True)
    plain = LSKNet_moe(embed_dims=[64, 128], depths=[1, 1], num_stages=2, mlp_ratios=[4, 4])
    pc = LskConfig(embed_dims=[64, 128], depths=[1, 1], num_stages=2, mlp_ratios=[4, 4], multi_input=False,
                   MoE_Block_inds_fc1=[[], []], MoE_Block_inds_fc2=[[], []])
    assert set(lsk_param_shapes(pc)) == set(plain.state_dict())
    with pytest.raises(RuntimeError):
        net(torch.zeros(1, 3, 64, 64))                    # CPU tensor: no fallback path
    ref = gen_reference_snapshots.load('lsk')['lsk_layout']
    assert ref['kw'] == kw
    assert set(ref['state_dict']) == set(sd)
    up = {k: torch.zeros(shape, dtype=dtype) for k, (shape, dtype) in ref['state_dict'].items()}
    assert not net.load_state_dict(up, strict=True).missing_keys


def test_lsk_upcycle_dense_checkpoint():
    from sm3det_b200 import LSKNet_moe
    dense = LSKNet_moe(embed_dims=[64, 128], depths=[1, 1], num_stages=2, mlp_ratios=[4, 4])
    moe = LSKNet_moe(embed_dims=[64, 128], depths=[1, 1], num_stages=2, mlp_ratios=[4, 4], num_experts=3, top_k=2,
                     MoE_Block_inds_fc1=[[], [0]], MoE_Block_inds_fc2=[[0], []])
    up = moe.upcycle_state_dict(dense.state_dict())
    res = moe.load_state_dict(up, strict=False)
    assert not res.unexpected_keys
    assert all('w_gate' in k or 'w_noise' in k or k.endswith(('.mean', '.std')) for k in res.missing_keys)
    for e in range(3):
        assert torch.equal(moe.block2[0].mlp.fc1.experts[e].weight, dense.block2[0].mlp.fc1.weight)
        assert torch.equal(moe.block1[0].mlp.fc2.experts[e].bias, dense.block1[0].mlp.fc2.bias)


def test_lsk_multi_input_upcycle_moves_the_stem():
    """lsk_moe.py:806-813: a dense LSKNet checkpoint's 'patch_embed1.proj.*' must land in 'dataset_stems.single.*' and
    'patch_embed1.norm.*' in 'patch_embed1.*' (round-1 advisor finding: they were silently dropped)."""
    from sm3det_b200 import LSKNet_moe, LSKNet_moe_MultiInput
    kw = dict(embed_dims=[64, 128], depths=[1, 1], num_stages=2, mlp_ratios=[4, 4])
    dense = LSKNet_moe(**kw)
    with torch.no_grad():
        dense.patch_embed1.norm.running_mean.normal_()
    moe = LSKNet_moe_MultiInput(num_experts=3, top_k=2, MoE_Block_inds_fc1=[[], [0]], MoE_Block_inds_fc2=[[0], []], **kw)
    res = moe.load_state_dict(moe.upcycle_state_dict(dense.state_dict()), strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    assert all('w_gate' in k or 'w_noise' in k or k.endswith(('.mean', '.std')) for k in res.missing_keys), res.missing_keys
    assert torch.equal(moe.dataset_stems['single'].weight, dense.patch_embed1.proj.weight)
    assert torch.equal(moe.dataset_stems['single'].bias, dense.patch_embed1.proj.bias)
    assert torch.equal(moe.patch_embed1.weight, dense.patch_embed1.norm.weight)
    assert torch.equal(moe.patch_embed1.running_mean, dense.patch_embed1.norm.running_mean)
    for e in range(3):
        assert torch.equal(moe.block2[0].mlp.fc1.experts[e].weight, dense.block2[0].mlp.fc1.weight)


def test_lsk_init_weights_from_scratch():
    """init_cfg=None branch of init_weights (lsk_moe.py:476-490): Conv2d ~ N(0, 2/fan_out), biases 0, LayerNorm (1, 0)."""
    from sm3det_b200 import LSKNet_moe_MultiInput
    net = LSKNet_moe_MultiInput(embed_dims=[64, 128], depths=[1, 1], num_stages=2, mlp_ratios=[4, 4], init_cfg=None)
    with torch.no_grad():
        for p in net.parameters():
            p.fill_(3.0)
    net.init_weights()
    conv = net.patch_embed2.proj
    fan_out = conv.kernel_size[0] * conv.kernel_size[1] * conv.out_channels // conv.groups
    assert abs(conv.weight.std().item() - (2.0 / fan_out) ** 0.5) < 0.2 * (2.0 / fan_out) ** 0.5
    assert float(conv.bias.abs().max()) == 0.0
    assert torch.equal(net.norm1.weight, torch.ones_like(net.norm1.weight)) and float(net.norm1.bias.abs().max()) == 0.0


def test_van_contract():
    """VAN_moe(_MultiInput): same contract as LSKNet with the LKA gating unit (van_moe.py:319-333, :410, :590)."""
    from sm3det_b200 import build_backbone
    kw = dict(MoE_Block_inds_fc1=[[], [0], [0], []], MoE_Block_inds_fc2=[[], [0], [0], []], num_experts=2, top_k=1,
              embed_dims=[32, 64, 160, 256], depths=[1, 1, 2, 1])
    net = build_backbone(dict(type='VAN_moe_MultiInput', **kw))
    shapes = lsk_param_shapes(LskConfig(spatial_unit='lka', **kw))
    sd = net.state_dict()
    assert set(shapes) == set(sd) and all(tuple(sd[k].shape) == tuple(v) for k, v in shapes.items())
    ref = gen_reference_snapshots.load('lsk')['van_layout']
    assert ref['kw'] == kw and set(ref['keys']) == set(sd)


def test_forced_channel_argmax_is_identity_on_own_choice():
    """forced_amax with the oracle's own argmax reproduces outputs and gradients; forcing another channel moves the gradient
    of the max feature to that channel (the mechanism the GPU parity test relies on for near-tie flips)."""
    spec = LSK_CASES['lsk_mini_dense_eval']
    cfg = LskConfig(**spec['kw'])
    sd = make_state_dict(lsk_param_shapes(cfg), 0, True)
    n, h, w = spec['img']
    x = make_images(n, h, w, seed=1234)

    def run(forced):
        sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and 'running_' not in k and 'num_batches' not in k else v) for k, v in sd.items()}
        rec = []
        outs = lsk_backbone_forward(sdg, cfg, x, train=True, bn_state={}, forced_amax=forced, amax_record=rec)
        outs = outs[0] if isinstance(outs[0], (tuple, list)) else outs
        sum(o.square().sum() for o in outs).backward()
        return outs, sdg, rec
    o_p, sd_p, rec = run(None)
    assert len(rec) == sum(cfg.depths) and all(float(r['gap'].abs().max()) == 0.0 for r in rec)
    o_f, sd_f, rec_f = run([r['own'] for r in rec])
    assert all(int((r['own'] != r['forced']).sum()) == 0 for r in rec_f)
    assert all(torch.equal(a, b) for a, b in zip(o_f, o_p))
    name = 'block1.0.attn.spatial_gating_unit.conv1.bias'
    assert torch.allclose(sd_f[name].grad, sd_p[name].grad, rtol=1e-5, atol=1e-9)
    _, sd_z, rec_z = run([torch.zeros_like(r['own']) for r in rec])
    assert float(rec_z[0]['gap'].max()) > 0.0
    assert not torch.allclose(sd_z[name].grad, sd_p[name].grad, rtol=1e-3)
