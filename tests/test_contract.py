"""CPU-side contract tests: the C-ABI library loads and exports everything the header declares, the module
tree reproduces the reference's state_dict layout / constructor surface, and the host logic around the
kernels (expert-parameter stacking, registry, bench reference arm under a 2-process launch) works."""
import json
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from sm3det_b200 import _lib
    if not os.path.isfile(_lib.library_path()):
        subprocess.run(['make', '-j8'], cwd=ROOT, check=True)
    lib = _lib.load()
    header = open(os.path.join(ROOT, 'include', 'sm3det_b200.h')).read()
    declared = set(re.findall(r'\b(sm3_[a-z0-9_]+)\s*\(', header))
    assert declared, 'no declarations parsed'
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in include/sm3det_b200.h but not exported'
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert lib.sm3_abi_version() == 1


def test_ops_refuse_cpu_tensors():
    from sm3det_b200 import ops
    with pytest.raises(RuntimeError, match='CUDA'):
        ops.scale_rows(torch.zeros(4, 32))


def test_backbone_refuses_cpu_input():
    from sm3det_b200 import ConvNeXt_moe
    net = ConvNeXt_moe(arch=dict(depths=[1, 1, 1, 1], channels=[32, 64, 96, 128]))
    with pytest.raises(RuntimeError, match='CUDA'):
        net(torch.zeros(1, 3, 64, 64))


@pytest.mark.parametrize('kw,multi', [
    (dict(arch='tiny'), True),
    (dict(arch='tiny', MoE_Block_inds=[[], [], [0, 2, 4, 6, 8], [0, 2]], num_experts=8, top_k=2), True),
    (dict(arch='tiny', MoE_Block_inds=[[], [], [0, 2, 4, 6, 8], [0, 2]], num_experts=8, top_k=3), False),
    (dict(arch='base', MoE_Block_inds=[[], [0, 2], list(range(0, 27, 2)), [0, 2]], num_experts=8, top_k=2), True),
])
def test_state_dict_layout_matches_reference(kw, multi):
    from oracle import gen_reference_snapshots
    from oracle.convnext_moe_oracle import OracleConfig, param_shapes
    from sm3det_b200 import build_backbone
    name = 'ConvNeXt_moe_MultiInput' if multi else 'ConvNeXt_moe'
    with torch.device('meta'):
        net = build_backbone(dict(type=name, **kw))
    mine = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    assert mine == param_shapes(OracleConfig(multi_input=multi, **kw))
    if kw['arch'] == 'tiny':          # recorded from the reference for the tiny cases (it cannot be built on 'meta')
        ref, = [r for r in gen_reference_snapshots.load('convnext')['layouts'] if r['cls'] == name and r['kw'] == kw]
        assert mine == ref['state_dict']
        assert sorted(n for n, _ in net.named_parameters()) == sorted(ref['params'])


def test_convnext_da_state_dict_and_shared_gate_weights():
    """ConvNeXt_DA_MultiInput (convnext_moe_DA.py): same keys, order and parameter names as the reference, including its quirk
    of ONE gate MLP registered under fc.0 / fc.1 / fc.2; the literal config dict of local_configs/main_DA_*.py builds."""
    from oracle import gen_reference_snapshots
    from oracle.convnext_moe_oracle import OracleConfig, param_shapes
    from sm3det_b200 import build_backbone
    kw = dict(arch='tiny', drop_path_rate=0.1, datasets=None)
    net = build_backbone(dict(type='ConvNeXt_DA_MultiInput', **kw))
    okw = {k: v for k, v in kw.items() if k != 'datasets'}
    assert {k: tuple(v.shape) for k, v in net.state_dict().items()} == param_shapes(OracleConfig(da=True, **okw))
    da = net.stages[0][0].DA
    assert da.fc[0] is da.fc[1] is da.fc[2]
    names = [n for n, _ in net.named_parameters()]
    assert 'stages.0.0.DA.fc.0.0.weight' in names and 'stages.0.0.DA.fc.1.0.weight' not in names      # de-duplicated like the reference
    ref = gen_reference_snapshots.load('convnext')['da_layout']      # recorded from the reference for these kwargs
    assert ref['kw'] == kw
    assert list(net.state_dict()) == list(ref['state_dict'])
    assert names == ref['params']
    with pytest.raises(NotImplementedError):
        build_backbone(dict(type='ConvNeXt_DA_MultiInput', arch='tiny', datasets=['sar', 'rgb', 'ifr']))


def test_registry_builds_literal_sm3det_config_dicts():
    """The backbone dicts of configs/SM3Det/SM3Det_convnext_{t,b}.py, verbatim (minus init_cfg's checkpoint)."""
    from sm3det_b200 import ROTATED_BACKBONES, build_backbone
    t = dict(type='ConvNeXt_moe_MultiInput', MoE_Block_inds=[[], [], [0, 2, 4, 6, 8], [0, 2]], datasets=None,
             num_experts=8, top_k=3, arch='tiny', drop_path_rate=0.1, init_cfg=None)
    with torch.device('meta'):
        net = build_backbone(t)
    assert net.depths == [3, 3, 9, 3] and net.channels == [96, 192, 384, 768]
    assert sum(1 for m in net.modules() if m.__class__.__name__ == 'MoE_layer') == 7
    assert 'ConvNeXt_moe' in ROTATED_BACKBONES and 'ConvNeXt_moe_MultiInput' in ROTATED_BACKBONES
    with pytest.raises(TypeError, match='ConvNeXt_moe_MultiInput'):
        build_backbone(dict(type='ConvNeXt_moe_MultiInput', not_a_kwarg=1))
    with pytest.raises(NotImplementedError):
        build_backbone(dict(type='ConvNeXt_moe', arch='tiny', gate='linear', MoE_Block_inds=[[0], [], [], []]))
    net.train()
    assert net.get_layer_depth('backbone.stages.2.4.gamma', 'backbone.') == (4, 8)


def test_upcycling_maps_dense_checkpoint_keys():
    from sm3det_b200 import ConvNeXt_moe_MultiInput
    with torch.device('meta'):
        net = ConvNeXt_moe_MultiInput(arch=dict(depths=[1, 1, 2, 1], channels=[32, 64, 96, 128]),
                                      MoE_Block_inds=[[], [], [1], []], num_experts=3)
    src = {'backbone.downsample_layers.0.0.weight': 0, 'backbone.downsample_layers.0.1.bias': 1,
           'backbone.stages.2.1.pointwise_conv1.weight': 2, 'backbone.stages.2.0.pointwise_conv2.bias': 3,
           'backbone.stages.0.0.gamma': 4, 'neck.x': 5}
    out = net.upcycle_state_dict(src, multi_input=True)
    assert out['dataset_stems.single.weight'] == 0 and out['downsample_layers.0.0.bias'] == 1
    assert all(out[f'stages.2.1.ffn.experts.{e}.pointwise_conv1.weight'] == 2 for e in range(3))
    assert out['stages.2.0.ffn.pointwise_conv2.bias'] == 3 and out['stages.0.0.gamma'] == 4 and 'neck.x' not in out
    assert set(out) <= set(net.state_dict())


def test_stack_expert_params_keeps_parameter_identity():
    from sm3det_b200.functional import stack_expert_params
    ps = [torch.nn.Parameter(torch.randn(4, 3)) for _ in range(5)]
    vals = [p.detach().clone() for p in ps]
    ids = [id(p) for p in ps]
    stack_expert_params(ps)
    step = ps[0].numel() * 4
    assert all(p.data_ptr() == ps[0].data_ptr() + i * step for i, p in enumerate(ps))
    assert all(torch.equal(p, v) for p, v in zip(ps, vals)) and ids == [id(p) for p in ps]
    ptr = ps[0].data_ptr()
    stack_expert_params(ps)                      # already adjacent: no reallocation
    assert ps[0].data_ptr() == ptr
    with torch.no_grad():
        ps[2].add_(1.0)                          # in-place optimizer-style update stays visible in the stack
    assert torch.equal(ps[2], vals[2] + 1.0)


def test_reference_arm_two_processes_gloo_style_launch():
    """`bench.py --impl reference` under a 2-rank launch: rank 0 alone prints the JSON line."""
    env = dict(os.environ, MASTER_ADDR='127.0.0.1', MASTER_PORT='29533')
    outs = []
    for rank in (0, 1):
        e = dict(env, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE='2')
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2',
                            '--steps', '1', '--warmup', '0', '--size', '64', '--cpu-images', '1'],
                           env=e, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append(r.stdout.strip())
    assert outs[1] == ''
    line = json.loads(outs[0].splitlines()[-1])
    assert line['impl'] == 'reference' and line['cpu_baseline']['kind'] == 'port' and line['value'] > 0
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['unit'] == 'img/s'


def test_pack_cache_invalidation(monkeypatch):
    """PackCache re-splits a weight image exactly when a parameter changed in place (optimizer step / load_state_dict) or
    moved (stack_expert_params re-pointing .data) -- host logic, checked with a stub in place of the CUDA pack kernel."""
    import torch
    from sm3det_b200 import ops
    from sm3det_b200.backbone import PackCache
    calls = []

    def fake_pack(w, *, transposed, groups=1, out=None, tile=0):
        calls.append((w.data_ptr(), transposed, groups, tile))
        return (out if out is not None else torch.zeros(4, dtype=torch.int16)), 4

    monkeypatch.setattr(ops, 'pack_weight', fake_pack)
    pc = PackCache()
    p = torch.nn.Parameter(torch.randn(8, 8))
    a = pc.get('w1', [p], False)
    assert pc.get('w1', [p], False) is a and len(calls) == 1            # hit
    pc.get('w1', [p], True)
    assert len(calls) == 2                                               # the transposed image is a separate entry
    pc.get('w1', [p], False, tile=64)
    assert len(calls) == 3 and pc.get('w1', [p], False, tile=64) is not a  # so is an image with another tile width
    assert pc.get('w1', [p], False) is a
    calls.pop()
    with torch.no_grad():
        p.add_(1.0)                                                      # what an optimizer step does
    pc.get('w1', [p], False)
    assert len(calls) == 3
    p.data = p.data.clone()                                              # storage moved
    pc.get('w1', [p], False)
    assert len(calls) == 4
    opt = torch.optim.SGD([p], lr=0.1)
    p.grad = torch.ones_like(p)
    opt.step()
    pc.get('w1', [p], False)
    assert len(calls) == 5


def test_ep_expert_layout_host_plan():
    """expert_parallel._expert_layout: 128-row aligned expert segments per owner, source-major offsets, tile map."""
    from sm3det_b200.expert_parallel import _expert_layout
    cnt = [[5, 0, 130, 1], [0, 0, 127, 300]]          # cnt[source][expert], W = 2, E = 4 (2 experts per rank)
    seg, off, rows, tiles = _expert_layout(cnt, 2, 4)
    assert seg == [[0, 128], [0, 384]]                  # rank 0: e0 (5 rows -> 1 tile), e1 (0 rows -> 0 tiles at 128); rank 1: e2 257 rows -> 3 tiles, e3
    assert off[0] == [0, 5] and off[2] == [0, 130] and off[3] == [0, 1]
    assert rows == [128, 384 + 384]                     # e3: 301 rows -> 3 tiles
    assert tiles[0] == [0] and tiles[1] == [0, 0, 0, 1, 1, 1]


def test_bench_resolves_the_named_configs():
    """bench.py: the global batch of the named config is kept at every N (strong scaling), each GPU's share is one pass unless
    --micro-batch splits it, cfg4 turns expert parallelism on at N > 1, --batch switches to weak scaling."""
    import argparse
    import importlib.util
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    def ns(**kw):
        d = dict(config='t_e8', batch=None, global_batch=None, micro_batch=None, no_expert_parallel=False, expert_parallel=False, size=1024)
        d.update(kw)
        return argparse.Namespace(**d)
    for world, per in ((1, 32), (2, 16), (4, 8), (8, 4)):
        c, p, micro, scaling, ep = bench.resolve(ns(), world)
        assert (p, micro, scaling, ep) == (per, per, 'strong', False)
    assert bench.resolve(ns(micro_batch=8), 1)[1:3] == (32, 8)
    assert bench.resolve(ns(micro_batch=5), 1)[2] == 4                      # largest divisor of the share not above the request
    assert bench.resolve(ns(batch=8), 4)[1:4] == (8, 8, 'weak')
    assert bench.resolve(ns(config='b_e16'), 8)[4] is True and bench.resolve(ns(config='b_e16'), 1)[4] is False
    assert bench.resolve(ns(config='lsk_s'), 4)[1:3] == (4, 4)
    with pytest.raises(SystemExit):
        bench.resolve(ns(global_batch=30), 8)
    cfg = bench.workload_config(ns(), 8)
    assert cfg['global_batch'] == 32 and cfg['per_gpu_batch'] == 4 and cfg['parallelism'] == 'dp8' and cfg['noisy_gating'] is True
