"""Record what the tests compare against the UNMODIFIED reference into tests/golden/reference/*.pt.gz.

Run where the reference tree is available (see oracle/ref_shim.py):  python -m oracle.gen_reference_snapshots
The tests then need no reference checkout.  What is recorded:
  convnext  reference forward outputs of the ConvNeXt-MoE classes (tests/test_oracle.py) and the state_dict / parameter
            layouts of the ConvNeXt classes (tests/test_contract.py)
  lsk       LSKNet-MoE forward outputs and the LSKNet / VAN state_dict layouts (tests/test_lsk_oracle.py)
  fpn       MultitaskFPN state_dict keys and outputs (tests/test_fpn.py)
Outputs are kept as summarize_grad digests (every element of a small tensor; a fixed sample plus the full tensor's L2 norm
and sum of a larger one).  Every recorded output is also asserted bit-exact against the oracle here.
"""
import gzip
import io
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_shim                                                     # noqa: E402
from oracle.cases import CASES, GOLDEN_THREADS, LSK_CASES, summarize_grad       # noqa: E402
from oracle.convnext_moe_oracle import OracleConfig, backbone_forward, param_shapes  # noqa: E402
from oracle.fpn_oracle import fpn_forward, fpn_param_shapes                     # noqa: E402
from oracle.lsk_moe_oracle import LskConfig, lsk_backbone_forward, lsk_param_shapes  # noqa: E402
from sm3det_b200.synth import make_images, make_state_dict                      # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden', 'reference')
SAMPLES = 256

# (class, constructor kwargs) of the ConvNeXt layout checks in tests/test_contract.py that the reference can build
CONVNEXT_LAYOUTS = [
    ('ConvNeXt_moe_MultiInput', dict(arch='tiny')),
    ('ConvNeXt_moe_MultiInput', dict(arch='tiny', MoE_Block_inds=[[], [], [0, 2, 4, 6, 8], [0, 2]], num_experts=8, top_k=2)),
    ('ConvNeXt_moe', dict(arch='tiny', MoE_Block_inds=[[], [], [0, 2, 4, 6, 8], [0, 2]], num_experts=8, top_k=3)),
]
DA_KW = dict(arch='tiny', drop_path_rate=0.1, datasets=None)
PLAIN_KW = dict(arch=dict(depths=[1, 1, 2, 1], channels=[32, 64, 96, 128]), MoE_Block_inds=[[], [], [1], []], num_experts=4,
                top_k=2)
LSK_KW = dict(MoE_Block_inds_fc1=[[], [0], [0, 2], [0]], MoE_Block_inds_fc2=[[], [0], [0, 2], [0]], num_experts=4, top_k=2,
              embed_dims=[64, 128, 320, 512], depths=[2, 2, 4, 2], drop_rate=0.1, drop_path_rate=0.,
              norm_cfg=dict(type='SyncBN', requires_grad=True))
VAN_KW = dict(MoE_Block_inds_fc1=[[], [0], [0], []], MoE_Block_inds_fc2=[[], [0], [0], []], num_experts=2, top_k=1,
              embed_dims=[32, 64, 160, 256], depths=[1, 1, 2, 1])
FPN_KW = dict(in_channels=[96, 192, 384, 768], out_channels=256, extra_level=1, add_extra_convs='on_output', num_outs=5)


def load(name):
    """The recorded snapshot `name` (convnext | lsk | fpn)."""
    with open(os.path.join(OUT, name + '.pt.gz'), 'rb') as f:
        return torch.load(io.BytesIO(gzip.decompress(f.read())), weights_only=False)


def digest(ts):
    return [summarize_grad(t, full_below=SAMPLES, samples=SAMPLES) for t in ts]


def assert_equal(ref, orc):
    assert len(ref) == len(orc)
    for a, b in zip(ref, orc):
        assert torch.equal(a, b), f'oracle differs from the reference by {(a - b).abs().max()}'


def layout(net):
    return dict(state_dict={k: tuple(v.shape) for k, v in net.state_dict().items()},
                params=[n for n, _ in net.named_parameters()])


def convnext():
    snap = dict(live={}, layouts=[])
    for name in ('mini_moe_e4k2_eval', 'mini_moe_e8k3_eval'):
        kw = dict(CASES[name]['kw'])
        cfg = OracleConfig(**kw)
        net = ref_shim.build_reference_backbone('ConvNeXt_moe_MultiInput', seed=0, **kw)
        sd = make_state_dict(param_shapes(cfg), 3, True)
        net.load_state_dict(sd, strict=True)
        net.eval()
        x = make_images(2, 64, 64, seed=5)
        with torch.no_grad():
            (outs, loss), (o_outs, o_loss) = net(x), backbone_forward(sd, cfg, x)
        assert_equal(outs, o_outs)
        assert torch.equal(loss, o_loss)
        snap['live'][name] = dict(outs=digest(outs), gate_loss=loss.clone())
    cfg = OracleConfig(multi_input=False, **PLAIN_KW)
    net = ref_shim.build_reference_backbone('ConvNeXt_moe', seed=0, **PLAIN_KW)
    sd = make_state_dict(param_shapes(cfg), 1, True)
    net.load_state_dict(sd, strict=True)
    net.eval()
    x = make_images(1, 64, 64, seed=2)
    with torch.no_grad():
        outs, o_outs = net(x)[0], backbone_forward(sd, cfg, x)[0]
    assert_equal(outs, o_outs)
    snap['plain'] = dict(kw=PLAIN_KW, keys=sorted(net.state_dict()), outs=digest(outs))
    for cls, kw in CONVNEXT_LAYOUTS:
        snap['layouts'].append(dict(cls=cls, kw=kw, **layout(ref_shim.build_reference_backbone(cls, **kw))))
    da = ref_shim.build_reference_backbone('ConvNeXt_DA_MultiInput', module='convnext_moe_DA', **DA_KW)
    snap['da_layout'] = dict(kw=DA_KW, **layout(da))
    return snap


def lsk():
    spec = LSK_CASES['lsk_mini_moe_e4k2_eval']
    cfg = LskConfig(**spec['kw'])
    mod = ref_shim.load_reference_module('lsk_moe')
    torch.manual_seed(0)
    net = mod.LSKNet_moe_MultiInput(norm_cfg=dict(type='SyncBN', requires_grad=True), **spec['kw'])
    sd = make_state_dict(lsk_param_shapes(cfg), 0, True)
    net.load_state_dict(sd, strict=True)
    net.eval()
    x = make_images(*spec['img'], seed=5)
    with torch.no_grad():
        (outs, loss), (o_outs, o_loss) = net(x), lsk_backbone_forward(sd, cfg, x, train=False)
    assert_equal(outs, o_outs)
    assert torch.equal(loss, o_loss)
    ref = mod.LSKNet_moe_MultiInput(**LSK_KW)
    van = ref_shim.load_reference_module('van_moe').VAN_moe_MultiInput(**VAN_KW)
    return dict(live=dict(outs=digest(outs), gate_loss=loss.clone()),
                lsk_layout=dict(kw=LSK_KW, state_dict={k: (tuple(v.shape), v.dtype) for k, v in ref.state_dict().items()}),
                van_layout=dict(kw=VAN_KW, keys=sorted(van.state_dict())))


def fpn():
    mod = ref_shim.load_reference_module('Multitask_FPN', 'necks')
    ref = mod.MultitaskFPN(**FPN_KW)
    sd = make_state_dict(fpn_param_shapes(FPN_KW['in_channels'], 256, 5, 1, 'on_output'), 5, True)
    ref.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(3)
    xs = [torch.randn(2, c, 64 // (4 * 2 ** i), 64 // (4 * 2 ** i), generator=g) for i, c in enumerate(FPN_KW['in_channels'])]
    snap = dict(kw=FPN_KW, keys=sorted(ref.state_dict()), outs={})
    for start_level in (0, 1):
        with torch.no_grad():
            r = ref(xs, start_level=start_level, add_extra_convs='on_output') if start_level else ref(xs)
            o = fpn_forward(sd, xs, 4, 5, start_level, 'on_output')
        assert_equal(r, o)
        snap['outs'][start_level] = digest(r)
    return snap


if __name__ == '__main__':
    if not ref_shim.reference_available():
        raise SystemExit(f'reference tree not found under {ref_shim.REFERENCE_ROOT} (set SM3DET_REFERENCE_ROOT)')
    torch.set_num_threads(GOLDEN_THREADS)
    os.makedirs(OUT, exist_ok=True)
    for name, fn in (('convnext', convnext), ('lsk', lsk), ('fpn', fpn)):
        buf = io.BytesIO()
        torch.save(fn(), buf)
        path = os.path.join(OUT, name + '.pt.gz')
        with open(path, 'wb') as f:
            f.write(gzip.compress(buf.getvalue(), mtime=0))
        print(f'{path}: {os.path.getsize(path) / 1024:.0f} KiB')
