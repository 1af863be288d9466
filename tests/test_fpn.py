"""MultitaskFPN (next row, SURVEY 8f rank 1): oracle pinned against the unmodified reference's recorded outputs (CPU,
oracle/gen_reference_snapshots.py), drop-in contract, and GPU parity of forward + every gradient (incl. the gradient flowing
back into the 4 backbone maps) for the three call patterns the detector uses (trisource_H1stage_R2stage_detector.py:158-167)."""
import pytest
import torch

from oracle import gen_reference_snapshots
from oracle.cases import assert_matches_summary, golden_threads
from oracle.fpn_oracle import fpn_forward, fpn_param_shapes
from sm3det_b200.synth import make_state_dict

KW = dict(in_channels=[96, 192, 384, 768], out_channels=256, extra_level=1, add_extra_convs='on_output', num_outs=5)   # SM3Det_convnext_t.py:22-28


def _inputs(n=2, s=64, seed=3, chans=KW['in_channels']):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(n, c, s // (4 * 2 ** i), s // (4 * 2 ** i), generator=g) for i, c in enumerate(chans)]


def _sd():
    return make_state_dict(fpn_param_shapes(KW['in_channels'], 256, 5, 1, 'on_output'), 5, True)


@pytest.mark.parametrize('start_level', [0, 1])
def test_fpn_oracle_matches_reference(start_level):
    ref = gen_reference_snapshots.load('fpn')
    assert ref['kw'] == KW
    sd = _sd()
    assert set(sd) == set(ref['keys'])
    xs = _inputs()
    with torch.no_grad(), golden_threads():
        o = fpn_forward(sd, xs, 4, 5, start_level, 'on_output')
    r = ref['outs'][start_level]
    assert len(r) == len(o) == 5      # start_level=1 (SAR): 3 pyramid levels + 2 stride-2 extra levels
    for i, (a, b) in enumerate(zip(o, r)):
        assert_matches_summary(a, b, f'level {i}')


def test_fpn_contract():
    from sm3det_b200.neck import ROTATED_NECKS
    net = ROTATED_NECKS.build(dict(type='MultitaskFPN', **KW))
    sd = _sd()
    assert set(net.state_dict()) == set(sd)
    net.load_state_dict(sd, strict=True)
    with pytest.raises(RuntimeError):
        net(_inputs())                      # CPU tensors: no fallback


@pytest.mark.gpu
@pytest.mark.parametrize('start_level', [0, 1])
def test_fpn_gpu_matches_oracle(start_level):
    from sm3det_b200.neck import MultitaskFPN
    sd = _sd()
    net = MultitaskFPN(**KW)
    net.load_state_dict(sd, strict=True)
    net = net.cuda()
    xs = _inputs(n=2, s=96)
    xc = [x.clone().requires_grad_(True) for x in xs]
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    want = fpn_forward(sdg, xc, 4, 5, start_level, 'on_output')
    xg = [x.cuda().requires_grad_(True) for x in xs]
    got = net(xg, start_level=start_level, add_extra_convs='on_output') if start_level else net(xg)
    assert len(got) == len(want)
    rel = lambda a, b: ((a.detach().cpu() - b.detach()).abs().max() / (b.detach().abs().max() + 1e-30)).item()
    assert all(g.is_contiguous() and g.shape == w.shape for g, w in zip(got, want))
    assert max(rel(g, w) for g, w in zip(got, want)) < 1e-4
    ups = [torch.randn(w.shape, generator=torch.Generator().manual_seed(40 + i)) / w.numel() ** 0.5 for i, w in enumerate(want)]
    sum((w * u).sum() for w, u in zip(want, ups)).backward()
    sum((g * u.cuda()).sum() for g, u in zip(got, ups)).backward()
    for name, p in net.named_parameters():
        if sdg[name].grad is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, name
            continue
        assert rel(p.grad, sdg[name].grad) < 5e-4, name
    for i in range(start_level, 4):
        assert rel(xg[i].grad, xc[i].grad) < 5e-4, i
