"""Drop-in ConvNeXt-MoE backbones running on the sm3det_b200 CUDA library.

Same class names, constructor kwargs, ``state_dict`` layout, forward signature and return
convention as the reference (mmrotate/models/backbones/convnext_moe.py):
  ConvNeXt_moe            :407-728     ConvNeXt_moe_MultiInput   :730-899
  ConvNeXtBlock           :295-379     FFN :381-405   MoE_layer :108-248   CosineTopKGate :88-106
  LayerNorm2d             :30-47
The sub-modules below are *parameter containers* with the reference's attribute names; all compute
goes through sm3det_b200.functional (NHWC fp32 end-to-end, NCHW only at the input and the 4 outputs).
"""
import math
from typing import Sequence

import torch
import torch.nn as nn

from . import functional as Fn
from .registry import ROTATED_BACKBONES, BaseModule

ARCH_SETTINGS = {
    'atto': dict(depths=[2, 2, 6, 2], channels=[40, 80, 160, 320]),
    'femto': dict(depths=[2, 2, 6, 2], channels=[48, 96, 192, 384]),
    'pico': dict(depths=[2, 2, 6, 2], channels=[64, 128, 256, 512]),
    'nano': dict(depths=[2, 2, 8, 2], channels=[80, 160, 320, 640]),
    'tiny': dict(depths=[3, 3, 9, 3], channels=[96, 192, 384, 768]),
    'small': dict(depths=[3, 3, 27, 3], channels=[96, 192, 384, 768]),
    'base': dict(depths=[3, 3, 27, 3], channels=[128, 256, 512, 1024]),
    'swin_large': dict(depths=[2, 2, 18, 2], channels=[192, 384, 768, 1536]),
    'large': dict(depths=[3, 3, 27, 3], channels=[192, 384, 768, 1536]),
    'xlarge': dict(depths=[3, 3, 27, 3], channels=[256, 512, 1024, 2048]),
    'huge': dict(depths=[3, 3, 27, 3], channels=[352, 704, 1408, 2816]),
}


class LayerNorm2d(nn.LayerNorm):
    """Parameter holder (weight, bias, eps); normalisation runs in sm3_layernorm_fwd."""

    def __init__(self, num_channels: int, **kwargs) -> None:
        super().__init__(num_channels, **kwargs)
        self.num_channels = self.normalized_shape[0]


def build_LayerNorm2d_layer(cfg: dict, num_features: int) -> nn.Module:
    if not isinstance(cfg, dict):
        raise TypeError('cfg must be a dict')
    if 'type' not in cfg:
        raise KeyError('the cfg dict must contain the key "type"')
    cfg_ = cfg.copy()
    cfg_.pop('type')
    requires_grad = cfg_.pop('requires_grad', True)
    cfg_.setdefault('eps', 1e-5)
    layer = LayerNorm2d(num_features, **cfg_)
    for param in layer.parameters():
        param.requires_grad = requires_grad
    return layer


class FFN(nn.Module):
    def __init__(self, in_channels, mid_channels):
        super().__init__()
        self.pointwise_conv1 = nn.Linear(in_channels, mid_channels)
        self.pointwise_conv2 = nn.Linear(mid_channels, in_channels)


class CosineTopKGate(nn.Module):
    def __init__(self, model_dim, num_global_experts, init_t=0.5):
        super().__init__()
        proj_dim = min(model_dim // 2, 256)
        self.temperature = nn.Parameter(torch.log(torch.full([1], 1.0 / init_t)), requires_grad=True)
        self.cosine_projector = nn.Linear(model_dim, proj_dim)
        self.sim_matrix = nn.Parameter(torch.randn(size=(proj_dim, num_global_experts)), requires_grad=True)
        nn.init.normal_(self.sim_matrix, 0, 0.01)


class MoE_layer(nn.Module):
    def __init__(self, in_channels, mid_channels, num_experts, top_k, noisy_gating, gating):
        super().__init__()
        if gating != 'cosine':
            raise NotImplementedError(
                "sm3det_b200: only gate='cosine' is implemented (gate='linear' starts from an all-zero w_gate, "
                'i.e. fully tied logits whose routing is implementation-defined in the reference)')
        assert top_k <= num_experts
        self.noisy_gating = noisy_gating
        self.num_experts = num_experts
        self.input_size = in_channels
        self.k = top_k
        self.gating = gating
        self.experts = nn.ModuleList([FFN(in_channels, mid_channels) for _ in range(num_experts)])
        self.w_gate = CosineTopKGate(in_channels, num_experts)
        self.w_noise = nn.Parameter(torch.zeros(in_channels, num_experts), requires_grad=True)
        self.register_buffer('mean', torch.tensor([0.0]))
        self.register_buffer('std', torch.tensor([1.0]))

    def expert_params(self):
        e = self.experts
        w1 = [m.pointwise_conv1.weight for m in e]
        b1 = [m.pointwise_conv1.bias for m in e]
        w2 = [m.pointwise_conv2.weight for m in e]
        b2 = [m.pointwise_conv2.bias for m in e]
        for group in (w1, b1, w2, b2):
            Fn.stack_expert_params(group)
        return w1 + b1 + w2 + b2


class PackCache:
    """Per-module cache of the pre-split (bf16 hi/lo, tile-ordered) weight images the GEMM bulk-copies.

    An entry is rebuilt when any of its parameters changed in place (tensor version counters, which every
    optimizer step / load_state_dict bumps) or moved (data_ptr, device); it lives and dies with the owning module.
    Writes that bypass the version counter (``p.data.copy_()``, EMA swaps through ``.data``) need an explicit
    ``invalidate()`` -- ``ConvNeXtBlock._apply`` / ``load_state_dict`` hooks call it for the common cases.
    """

    def __init__(self):
        self._d = {}

    def invalidate(self):
        self._d.clear()

    def get(self, name, params, transposed, tile=0):
        from . import ops
        key = tuple(p._version for p in params) + (params[0].data_ptr(), str(params[0].device))
        name = (name, tile)
        hit = self._d.get((name, transposed))
        if hit is not None and hit[0] == key:
            return hit[1]
        reuse = None if hit is None or hit[1][0].device != params[0].device else hit[1][0]   # never write into a buffer
        with torch.no_grad():                                                                # left behind on another GPU
            packed = ops.pack_weight(params[0], transposed=transposed, groups=len(params), out=reuse, tile=tile)
        self._d[(name, transposed)] = (key, packed)
        return packed


class ConvNeXtBlock(nn.Module):
    def __init__(self, in_channels, norm_cfg, mlp_ratio=4., MoE_cfg=None, drop_path_rate=0.,
                 layer_scale_init_value=1e-6):
        super().__init__()
        self.depthwise_conv = nn.Conv2d(in_channels, in_channels, groups=in_channels, kernel_size=7, padding=3)
        self.norm = build_LayerNorm2d_layer(norm_cfg, in_channels)
        mid = int(mlp_ratio * in_channels)
        self.MoE_cfg = MoE_cfg
        if MoE_cfg is not None:
            self.ffn = MoE_layer(in_channels, mid, MoE_cfg['num_experts'], MoE_cfg['top_k'], MoE_cfg['noisy_gating'],
                                 MoE_cfg['gating'])
        else:
            self.ffn = FFN(in_channels, mid)
        if not layer_scale_init_value > 0:
            raise NotImplementedError('sm3det_b200: layer_scale_init_value must be > 0 (gamma is fused in the epilogue)')
        self.gamma = nn.Parameter(layer_scale_init_value * torch.ones((in_channels)), requires_grad=True)
        self.drop_path_rate = float(drop_path_rate)
        self._packs = PackCache()

    def _apply(self, fn, recurse=True):      # .to() / .cuda() / .half(): cached images no longer describe the weights
        self._packs.invalidate()
        return super()._apply(fn, recurse)

    def _load_from_state_dict(self, *args, **kwargs):
        self._packs.invalidate()
        return super()._load_from_state_dict(*args, **kwargs)

    def forward(self, x, record=None):
        """x: NHWC fp32.  Returns (x, loss) like the reference block (:343-379); loss is None if dense."""
        return self._run(x, Fn.drop_path_row_scale(self, x), record, True)

    def _run(self, x, rs, record, shortcut):
        """shortcut=False returns the branch rs * gamma * ffn(norm(dwconv(x))) without the residual add (ConvNeXt_DA)."""
        eps = self.norm.eps
        dw = self.depthwise_conv
        grad = torch.is_grad_enabled()
        pc = self._packs
        from . import ops
        if self.MoE_cfg is None:
            f = self.ffn
            w1, w2 = f.pointwise_conv1.weight, f.pointwise_conv2.weight
            C = w2.shape[0]
            cf = ops.ffn_chunk(0, C)
            if cf > 0:
                # fused FFN forward: weight images in the chunk widths the kernel streams (csrc/ffn_fused.cu)
                packs = {'fused': dict(fwd=cf), 'w1_c': pc.get('w1', [w1], False, tile=cf), 'w2_n': pc.get('w2', [w2], False, tile=C)}
            else:
                packs = {'w1': pc.get('w1', [w1], False), 'w2': pc.get('w2', [w2], False)}
            if grad:
                packs['w1_t'] = pc.get('w1', [w1], True)
            packs['grad'] = grad
            packs['shortcut'] = shortcut
            out = Fn.DenseBlockFn.apply(x, dw.weight, dw.bias, self.norm.weight, self.norm.bias,
                                        w1, f.pointwise_conv1.bias, w2, f.pointwise_conv2.bias, self.gamma, rs, eps, packs)
            return out, None
        m = self.ffn
        noise = Fn.gating_noise(m, x.shape[0] * x.shape[1] * x.shape[2], x.device)
        g = m.w_gate
        ep = m.expert_params()
        E = m.num_experts
        w1s, w2s = ep[0:E], ep[2 * E:3 * E]
        epc = getattr(self, '_ep', None)
        if epc is not None:
            # expert parallel (sm3det_b200.expert_parallel): this rank only packs / runs the experts it owns
            if not shortcut:
                raise NotImplementedError('sm3det_b200: expert parallelism is not wired for the ConvNeXt_DA blocks')
            from .expert_parallel import EPMoEBlockFn
            El = E // epc.world
            o1, o2 = w1s[epc.rank * El:(epc.rank + 1) * El], w2s[epc.rank * El:(epc.rank + 1) * El]
            packs = {'w1': pc.get('w1', o1, False), 'w2': pc.get('w2', o2, False)}
            if grad:
                packs['w1_t'] = pc.get('w1', o1, True)
                packs['w2_t'] = pc.get('w2', o2, True)
                packs['wp_t'] = pc.get('wp', [g.cosine_projector.weight], True)
            return EPMoEBlockFn.apply(x, dw.weight, dw.bias, self.norm.weight, self.norm.bias, self.gamma,
                                      g.cosine_projector.weight, g.cosine_projector.bias, g.sim_matrix, g.temperature,
                                      m.w_noise, rs, noise, eps, E, m.k, record, packs, epc, self._ep_key, *ep)
        packs = {'w1': pc.get('w1', w1s, False), 'w2': pc.get('w2', w2s, False)}
        if grad:
            packs['w1_t'] = pc.get('w1', w1s, True)
            packs['w2_t'] = pc.get('w2', w2s, True)
            packs['wp_t'] = pc.get('wp', [g.cosine_projector.weight], True)
        packs['shortcut'] = shortcut
        out, loss = Fn.MoEBlockFn.apply(x, dw.weight, dw.bias, self.norm.weight, self.norm.bias, self.gamma,
                                        g.cosine_projector.weight, g.cosine_projector.bias, g.sim_matrix, g.temperature,
                                        m.w_noise, rs, noise, eps, E, m.k, record, packs, *ep)
        return out, loss


class DALayer(nn.Module):
    """Per-dataset squeeze-and-excitation gate (convnext_moe_DA.py:295-319).  The module tree repeats the reference's:
    ``fc`` is a ModuleList holding the SAME Sequential three times (`[...] * 3`, :299-304), so the state_dict lists one pair
    of weights under fc.0 / fc.1 / fc.2 and the three datasets share them."""
    dataset_DA = {'sar': 0, 'rgb': 1, 'ifr': 2}

    def __init__(self, channel, reduction=16):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool2d(1)
        self.fc = nn.ModuleList([nn.Sequential(nn.Linear(channel, channel // reduction, bias=False), nn.ReLU(inplace=True),
                                               nn.Linear(channel // reduction, channel, bias=False), nn.Sigmoid())] * 3)

    def gate(self, m, datasets):
        """m: [N, C] per-sample means of the branch -> [N, C] gates.  [N,C]-sized glue in torch (fp32 also under autocast)."""
        with torch.autocast('cuda', enabled=False):
            if len(datasets) == 1:
                return self.fc[self.dataset_DA[datasets[0]]](m)
            if len(datasets) != m.shape[0]:
                raise ValueError(f'ConvNeXt_DA: {len(datasets)} dataset names for a batch of {m.shape[0]} (the reference zips them '
                                 f'sample by sample, convnext_moe_DA.py:315-318)')
            return torch.cat([self.fc[self.dataset_DA[d]](row.view(1, -1)) for row, d in zip(m, datasets)], dim=0)


class ConvNeXtDABlock(ConvNeXtBlock):
    """ConvNeXtBlock whose branch is gated by a DALayer before drop-path and the shortcut (convnext_moe_DA.py:372-403)."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.avg_pool = nn.AdaptiveAvgPool2d(1)            # unused by the reference's forward too (:368); no parameters
        self.DA = DALayer(self.gamma.shape[0])

    def forward(self, x, record=None, datasets=('rgb',)):
        rs = Fn.drop_path_row_scale(self, x)
        y, loss = self._run(x, None, record, False)        # gamma * ffn(norm(dwconv(x))), NHWC
        s = self.DA.gate(Fn.SampleMeanFn.apply(y), list(datasets))
        return Fn.DAGateFn.apply(y, x, s, rs), loss


@ROTATED_BACKBONES.register_module()
class ConvNeXt_moe(BaseModule):
    arch_settings = ARCH_SETTINGS
    block_cls = ConvNeXtBlock

    def __init__(self, arch='tiny', in_channels=3, stem_patch_size=4, norm_cfg=dict(type='LN2d', eps=1e-6),
                 act_cfg=dict(type='GELU'), linear_pw_conv=True, use_grn=False, drop_path_rate=0.,
                 layer_scale_init_value=1e-6, out_indices=[0, 1, 2, 3], MoE_Block_inds=[[], [], [], []],
                 noisy_gating=True, num_experts=2, gate='cosine', top_k=2, frozen_stages=0,
                 gap_before_final_norm=False, with_cp=False,
                 init_cfg=[dict(type='TruncNormal', layer=['Conv2d', 'Linear'], std=.02, bias=0.),
                           dict(type='Constant', layer=['LayerNorm'], val=1., bias=0.)]):
        super().__init__(init_cfg=init_cfg)
        if isinstance(arch, str):
            assert arch in self.arch_settings, \
                f'Unavailable arch, please choose from ({set(self.arch_settings)}) or pass a dict.'
            arch = self.arch_settings[arch]
        elif isinstance(arch, dict):
            assert 'depths' in arch and 'channels' in arch, \
                f'The arch dict must have "depths" and "channels", but got {list(arch.keys())}.'
        if act_cfg.get('type', 'GELU') != 'GELU':
            raise NotImplementedError('sm3det_b200: only act_cfg=dict(type="GELU") is implemented')
        if not linear_pw_conv:
            raise NotImplementedError('sm3det_b200: linear_pw_conv=False (1x1 Conv2d FFN) is not implemented')
        if use_grn:
            raise NotImplementedError('sm3det_b200: use_grn=True is not implemented (no SM3Det config enables it)')
        if gap_before_final_norm:
            raise NotImplementedError('sm3det_b200: gap_before_final_norm=True is not implemented')
        self.depths = list(arch['depths'])
        self.channels = list(arch['channels'])
        assert (isinstance(self.depths, Sequence) and isinstance(self.channels, Sequence)
                and len(self.depths) == len(self.channels))
        for c in self.channels:
            if c % 32 != 0 or c > 1024:
                raise NotImplementedError(f'sm3det_b200: channel count {c} unsupported (multiple of 32, <= 1024)')
        self.num_stages = len(self.depths)
        if isinstance(out_indices, int):
            out_indices = [out_indices]
        out_indices = list(out_indices)
        for i, index in enumerate(out_indices):
            if index < 0:
                out_indices[i] = 4 + index
                assert out_indices[i] >= 0, f'Invalid out_indices {index}'
        self.out_indices = out_indices
        self.MoE_Block_inds = MoE_Block_inds
        self.num_experts = num_experts
        self.frozen_stages = frozen_stages
        self.gap_before_final_norm = gap_before_final_norm
        self.with_cp = with_cp     # activation checkpointing is not needed at 180 GB; accepted and ignored
        self.stem_patch_size = stem_patch_size
        self.norm_eps = norm_cfg.get('eps', 1e-5)

        dpr = [x.item() for x in torch.linspace(0, drop_path_rate, sum(self.depths), device='cpu')]
        block_idx = 0
        self.downsample_layers = nn.ModuleList()
        stem = nn.Sequential(
            nn.Conv2d(in_channels, self.channels[0], kernel_size=stem_patch_size, stride=stem_patch_size),
            build_LayerNorm2d_layer(norm_cfg, self.channels[0]))
        self.downsample_layers.append(stem)
        self.stages = nn.ModuleList()
        for i in range(self.num_stages):
            depth = self.depths[i]
            channels = self.channels[i]
            if i >= 1:
                self.downsample_layers.append(nn.Sequential(
                    build_LayerNorm2d_layer(norm_cfg, self.channels[i - 1]),
                    nn.Conv2d(self.channels[i - 1], channels, kernel_size=2, stride=2)))
            moe_ind = [list(range(depth))[q] for q in self.MoE_Block_inds[i] if q < depth]
            stage = nn.Sequential(*[
                self.block_cls(in_channels=channels, drop_path_rate=dpr[block_idx + j], norm_cfg=norm_cfg,
                              MoE_cfg={'noisy_gating': noisy_gating, 'num_experts': num_experts, 'top_k': top_k,
                                       'gating': gate} if j in moe_ind else None,
                              layer_scale_init_value=layer_scale_init_value) for j in range(depth)])
            block_idx += depth
            self.stages.append(stage)
            if i in self.out_indices:
                self.add_module(f'norm{i}', build_LayerNorm2d_layer(norm_cfg, channels))
        self._init_like_reference()
        self._freeze_stages()

    def _init_like_reference(self):
        """The reference never runs init_cfg (init_weights() only supports 'Pretrained'); weights stay at
        torch defaults.  We keep torch's default constructors too, so nothing to do."""

    # ---- forward -------------------------------------------------------------------------------
    def _stem(self, x):
        conv, ln = self.downsample_layers[0][0], self.downsample_layers[0][1]
        return Fn.StemFn.apply(x, conv.weight, conv.bias, ln.weight, ln.bias, ln.eps, self.stem_patch_size)

    def _trunk(self, x, record=None, datasets=None):
        outs, gate_losses = [], []
        for i, stage in enumerate(self.stages):
            if i >= 1:
                ln, conv = self.downsample_layers[i][0], self.downsample_layers[i][1]
                x = Fn.DownsampleFn.apply(x, ln.weight, ln.bias, conv.weight, conv.bias, ln.eps)
            for blk in stage:
                x, gate_loss = blk(x, record) if datasets is None else blk(x, record, datasets)
                if gate_loss is not None:
                    gate_losses.append(gate_loss)
            if i in self.out_indices:
                nl = getattr(self, f'norm{i}')
                outs.append(Fn.OutNormFn.apply(x, nl.weight, nl.bias, nl.eps))
        if len(gate_losses) > 0:
            return tuple(outs), sum(gate_losses) / len(gate_losses)
        return tuple(outs)

    def forward(self, x, record=None):
        self._check_input(x)
        with self._precision():
            return self._trunk(self._stem(x), record)

    def _precision(self):
        """Mixed-precision recipe (configs train with fp16=dict(loss_scale='dynamic')): under torch.autocast, or with
        ``self.amp = True``, the tensor-core GEMMs of this forward AND of its backward (ops.captures_precision) run
        single-pass bf16 (fp32 accumulation); router, LayerNorm, depthwise conv and combine stay fp32 like the
        reference's autocast policy.  The mode is scoped to this call, not a process global."""
        from . import ops
        return ops.precision_scope(ops.autocast_passes(self))

    @staticmethod
    def _check_input(x):
        if not x.is_cuda:
            raise RuntimeError('sm3det_b200 backbones run on CUDA (sm_100a) only; there is no CPU path')
        if x.dim() != 4 or x.shape[2] % 32 != 0 or x.shape[3] % 32 != 0:
            raise ValueError(f'expected [N,3,H,W] with H, W multiples of 32 (Pad size_divisor=32), got {tuple(x.shape)}')

    def _freeze_stages(self):
        for i in range(self.frozen_stages):
            downsample_layer = self.downsample_layers[i]
            stage = self.stages[i]
            downsample_layer.eval()
            stage.eval()
            for param in list(downsample_layer.parameters()) + list(stage.parameters()):
                param.requires_grad = False

    def train(self, mode=True):
        super().train(mode)
        self._freeze_stages()
        return self          # the reference returns None (:612-614); returning self is a harmless superset

    def get_layer_depth(self, param_name: str, prefix: str = ''):
        """Layer-wise depth of a parameter for layer-decay optimizers (:616-658)."""
        max_layer_id = 12 if self.depths[-2] > 9 else 6
        if not param_name.startswith(prefix):
            return max_layer_id + 1, max_layer_id + 2
        param_name = param_name[len(prefix):]
        if param_name.startswith('downsample_layers'):
            stage_id = int(param_name.split('.')[1])
            if stage_id == 0:
                layer_id = 0
            elif stage_id == 1 or stage_id == 2:
                layer_id = stage_id + 1
            else:
                layer_id = max_layer_id
        elif param_name.startswith('stages'):
            stage_id = int(param_name.split('.')[1])
            block_id = int(param_name.split('.')[2])
            if stage_id == 0 or stage_id == 1:
                layer_id = stage_id + 1
            elif stage_id == 2:
                layer_id = 3 + block_id // 3
            else:
                layer_id = max_layer_id
        else:
            layer_id = max_layer_id + 1
        return layer_id, max_layer_id + 2

    # ---- checkpoint up-cycling (:660-727, :824-899) --------------------------------------------
    def upcycle_state_dict(self, src, multi_input=False):
        """Map a dense ConvNeXt detector checkpoint onto this module's keys: strip 'backbone.', copy each
        dense pointwise_conv{1,2} into every expert of the MoE blocks, move the stem for MultiInput."""
        out = {}
        for k, v in src.items():
            if not k.startswith('backbone.'):
                continue
            k = k[9:]
            if multi_input and 'downsample_layers.0.0' in k:
                out[k.replace('downsample_layers.0.0', 'dataset_stems.single')] = v
            elif multi_input and 'downsample_layers.0.1' in k:
                out[k.replace('downsample_layers.0.1', 'downsample_layers.0.0')] = v
            elif 'pointwise_conv' in k:
                parts = k.split('.')
                stage_ind, block_ind = int(parts[1]), int(parts[2])
                if block_ind in self.MoE_Block_inds[stage_ind]:
                    for e in range(self.num_experts):
                        out[k.replace('pointwise_conv', f'ffn.experts.{e}.pointwise_conv')] = v
                else:
                    out[k.replace('pointwise_conv', 'ffn.pointwise_conv')] = v
            else:
                out[k] = v
        if out and next(iter(out)).startswith('module.'):
            out = {k[7:]: v for k, v in out.items()}
        return out

    def init_weights(self):
        cfg = self.init_cfg
        if isinstance(cfg, dict) and cfg.get('type') == 'Pretrained' and cfg.get('checkpoint'):
            ckpt = torch.load(cfg['checkpoint'], map_location='cpu')
            sd = ckpt.get('state_dict', ckpt.get('model', ckpt))
            sd = self.upcycle_state_dict(sd, multi_input=isinstance(self, ConvNeXt_moe_MultiInput))
            print(self.load_state_dict(sd, strict=False))
        # any other init_cfg: the reference constructor's own initialisation already ran


@ROTATED_BACKBONES.register_module()
class ConvNeXt_moe_MultiInput(ConvNeXt_moe):
    def __init__(self, arch='tiny', in_channels=3, stem_patch_size=4, datasets=None,
                 norm_cfg=dict(type='LN2d', eps=1e-6), act_cfg=dict(type='GELU'), linear_pw_conv=True,
                 use_grn=False, drop_path_rate=0., layer_scale_init_value=1e-6, out_indices=[0, 1, 2, 3],
                 MoE_Block_inds=[[], [], [], []], noisy_gating=True, num_experts=2, top_k=2, gate='cosine',
                 frozen_stages=0, gap_before_final_norm=False, with_cp=False,
                 init_cfg=[dict(type='TruncNormal', layer=['Conv2d', 'Linear'], std=.02, bias=0.),
                           dict(type='Constant', layer=['LayerNorm'], val=1., bias=0.)]):
        super().__init__(MoE_Block_inds=MoE_Block_inds, noisy_gating=noisy_gating, num_experts=num_experts,
                         gate=gate, top_k=top_k, arch=arch, in_channels=in_channels,
                         stem_patch_size=stem_patch_size, norm_cfg=norm_cfg, act_cfg=act_cfg,
                         linear_pw_conv=linear_pw_conv, use_grn=use_grn, drop_path_rate=drop_path_rate,
                         layer_scale_init_value=layer_scale_init_value, out_indices=out_indices,
                         frozen_stages=frozen_stages, gap_before_final_norm=gap_before_final_norm,
                         with_cp=with_cp, init_cfg=init_cfg)
        self.downsample_layers[0] = nn.Sequential(build_LayerNorm2d_layer(norm_cfg, self.channels[0]))
        self.datasets = ['single']
        self.dataset_stems = nn.ModuleDict()
        self.dataset_stems['single'] = nn.Conv2d(in_channels, self.channels[0], kernel_size=stem_patch_size,
                                                 stride=stem_patch_size)

    def _stem(self, x):
        conv, ln = self.dataset_stems['single'], self.downsample_layers[0][0]
        return Fn.StemFn.apply(x, conv.weight, conv.bias, ln.weight, ln.bias, ln.eps, self.stem_patch_size)

    def forward(self, x, datasets=['single'], record=None):
        if len(datasets) == 1:
            x = [x]
        x = torch.cat(list(x), dim=0)          # one shared stem for every modality (:798-801)
        self._check_input(x)
        with self._precision():
            return self._trunk(self._stem(x), record)


@ROTATED_BACKBONES.register_module()
class ConvNeXt_DA_MultiInput(ConvNeXt_moe_MultiInput):
    """convnext_moe_DA.py:762-860 (local_configs/main_DA_convnext_t_orcnn_gfl.py): ConvNeXt_moe_MultiInput whose every block
    carries a DALayer; `forward(x, datasets)` hands the dataset names to the blocks -- one name for the whole batch, or one
    name per sample (the detector passes one image per modality)."""
    block_cls = ConvNeXtDABlock

    def __init__(self, *args, datasets=None, **kwargs):
        super().__init__(*args, datasets=datasets, **kwargs)
        if datasets is not None and list(datasets) != ['single']:
            raise NotImplementedError('sm3det_b200: per-dataset stems (datasets=[...]) are not implemented; the reference forward '
                                      "only ever uses dataset_stems['single'] (convnext_moe_DA.py:836)")
        self.init_datasets = datasets

    def forward(self, x, datasets=['single'], record=None):
        if len(datasets) == 1:
            x = [x]
        x = torch.cat(list(x), dim=0)
        self._check_input(x)
        with self._precision():
            return self._trunk(self._stem(x), record, list(datasets))

    def init_weights(self):
        super().init_weights()
        cfg = self.init_cfg
        if isinstance(cfg, dict) and cfg.get('type') == 'Pretrained':
            for stage in self.stages:                      # :935-941: the gates start at sigmoid(0) = 0.5
                for blk in stage:
                    for m in range(3):
                        nn.init.constant_(blk.DA.fc[m][2].weight, 0.0)
