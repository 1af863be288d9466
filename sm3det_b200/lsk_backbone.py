"""Drop-in LSKNet-MoE backbones (BASELINE config 5) running on the sm3det_b200 CUDA library.

Same class names, constructor kwargs, ``state_dict`` layout, forward signature and return convention as the
reference (mmrotate/models/backbones/lsk_moe.py):
  LSKNet_moe :420-577        LSKNet_moe_MultiInput :600-826     Block :366-396      Attention :346-363
  LSKblock :319-343          Mlp :275-318   DWConv :580-587     OverlapPatchEmbed :399-418
  MoE_layer :80-228          CosineTopKGate :60-78              SparseDispatcher :230-273
The sub-modules are *parameter containers* with the reference's attribute names (so checkpoints load unchanged);
all compute goes through sm3det_b200.lsk_functional (NHWC fp32 end-to-end, NCHW only at the input image and the 4
returned feature maps).  ``norm_cfg=dict(type='SyncBN')`` all-reduces the batch statistics over the default process
group (NCCL) when one is initialised; at world size 1 it is plain BatchNorm, as in the reference.
"""
import math
import warnings
from functools import partial

import torch
import torch.nn as nn

from . import functional as Fn
from . import lsk_functional as LF
from .backbone import CosineTopKGate
from .registry import ROTATED_BACKBONES, BaseModule


def _build_bn(norm_cfg, dim):
    """build_norm_layer(norm_cfg, dim)[1] for BN / SyncBN (lsk_moe.py:369-374); returns (module, sync flag)."""
    if norm_cfg:
        t = norm_cfg.get('type', 'BN')
        if t not in ('BN', 'SyncBN', 'BN2d'):
            raise NotImplementedError(f'sm3det_b200: norm_cfg type {t!r} is not implemented for LSKNet (BN / SyncBN)')
        bn = nn.BatchNorm2d(dim, eps=norm_cfg.get('eps', 1e-5), momentum=norm_cfg.get('momentum', 0.1))
        for p in bn.parameters():
            p.requires_grad = norm_cfg.get('requires_grad', True)
        bn._sm3_sync = (t == 'SyncBN')
        return bn
    bn = nn.BatchNorm2d(dim)
    bn._sm3_sync = False
    return bn


def _bn(bn, x):
    train = bn.training or not bn.track_running_stats
    if train and bn.track_running_stats:
        bn.num_batches_tracked.add_(1)
    return LF.BatchNormFn.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, train, bn.momentum, bn.eps,
                                getattr(bn, '_sm3_sync', False))


def _conv1x1(conv, x, gelu=False):
    return LF.LinearFn.apply(x, conv.weight, conv.bias, gelu)


class MoE_layer(nn.Module):
    """lsk_moe.py:80-228.  Experts are single Conv2d(in, out, 1); input / output are NHWC here."""

    def __init__(self, moe_cfg):
        super().__init__()
        self.noisy_gating = moe_cfg['noisy_gating']
        self.num_experts = moe_cfg['num_experts']
        self.input_size = moe_cfg['in_channels']
        self.output_size = moe_cfg['out_channels']
        self.k = moe_cfg['top_k']
        self.gating = moe_cfg['gating']
        if self.gating != 'cosine':
            raise NotImplementedError("sm3det_b200: only gate='cosine' is implemented")
        if self.input_size % 32 or self.output_size % 32:
            raise NotImplementedError('sm3det_b200: MoE layer widths must be multiples of 32')
        self.experts = nn.ModuleList([nn.Conv2d(self.input_size, self.output_size, 1) for _ in range(self.num_experts)])
        self.infer_expert = None
        self.w_gate = CosineTopKGate(self.input_size, self.num_experts)
        self.w_noise = nn.Parameter(torch.zeros(self.input_size, self.num_experts), requires_grad=True)
        self.register_buffer('mean', torch.tensor([0.0]))
        self.register_buffer('std', torch.tensor([1.0]))
        assert self.k <= self.num_experts

    def expert_params(self):
        ws = [m.weight for m in self.experts]
        bs = [m.bias for m in self.experts]
        Fn.stack_expert_params(ws)
        Fn.stack_expert_params(bs)
        return ws + bs

    def forward(self, x, gamma=None, resid=None, row_scale=None, record=None):
        noise = Fn.gating_noise(self, x.numel() // x.shape[-1], x.device)
        g = self.w_gate
        return LF.MoELinearFn.apply(x, g.cosine_projector.weight, g.cosine_projector.bias, g.sim_matrix, g.temperature,
                                    self.w_noise, noise, gamma, resid, row_scale, self.num_experts, self.k, record,
                                    *self.expert_params())


class DWConv(nn.Module):
    def __init__(self, dim=768):
        super().__init__()
        self.dwconv = nn.Conv2d(dim, dim, 3, 1, 1, bias=True, groups=dim)


class Mlp(nn.Module):
    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0., MoE_cfg1=None,
                 MoE_cfg2=None):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        if act_layer is not nn.GELU:
            raise NotImplementedError('sm3det_b200: only act_layer=nn.GELU is implemented')
        self.MoE_cfg1, self.MoE_cfg2 = MoE_cfg1, MoE_cfg2
        if MoE_cfg1 is not None:
            MoE_cfg1.update({'in_channels': in_features, 'out_channels': hidden_features})
            self.fc1 = MoE_layer(MoE_cfg1)
        else:
            self.fc1 = nn.Conv2d(in_features, hidden_features, 1)
        if MoE_cfg2 is not None:
            MoE_cfg2.update({'in_channels': hidden_features, 'out_channels': out_features})
            self.fc2 = MoE_layer(MoE_cfg2)
        else:
            self.fc2 = nn.Conv2d(hidden_features, out_features, 1)
        self.dwconv = DWConv(hidden_features)
        self.act = act_layer()
        self.drop = nn.Dropout(drop)

    def _dropout(self, x):
        p = self.drop.p
        if p == 0.0 or not self.training:
            return x
        masks = getattr(self, '_injected_drop_masks', None)
        if masks:                                   # tests inject the reference's masks
            m = masks.pop(0).to(x.device, torch.float32).reshape(x.shape).contiguous()
            return LF.MulFn.apply(x, m)
        if torch.cuda.is_current_stream_capturing():
            seed = torch.randint(0, 2 ** 62, (1,), device=x.device)     # graph-safe: drawn on the device at every replay
        else:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())          # host RNG (torch.manual_seed reproducible), no device sync
        return LF.DropoutFn.apply(x, p, seed)

    def forward(self, x, ls, resid, row_scale, record=None):
        """x: NHWC BN output.  Returns (resid + row_scale * ls * mlp(x), loss or None)  (Block.forward :390-395)."""
        loss = []
        if self.MoE_cfg1 is not None:
            x, l1 = self.fc1(x, record=record)
            loss.append(l1)
        else:
            x = _conv1x1(self.fc1, x)
        dw = self.dwconv.dwconv
        x = LF.DWConvFn.apply(x, dw.weight, dw.bias, 3, 1)
        x = LF.GeluFn.apply(x)
        x = self._dropout(x)
        final_drop = self.drop.p > 0.0 and self.training
        if self.MoE_cfg2 is not None:
            if final_drop:
                x, l2 = self.fc2(x, record=record)
            else:
                out, l2 = self.fc2(x, gamma=ls, resid=resid, row_scale=row_scale, record=record)   # layer scale + shortcut fused
            loss.append(l2)
        else:
            x = _conv1x1(self.fc2, x)
        if self.MoE_cfg2 is None or final_drop:
            x = self._dropout(x)
            out = LF.AxpyFn.apply(x, resid, ls, row_scale)
        return out, (sum(loss) / len(loss) if loss else None)


class LSKblock(nn.Module):
    def __init__(self, dim):
        super().__init__()
        if dim % 64:
            raise NotImplementedError(f'sm3det_b200: LSKNet width {dim} unsupported (multiple of 64)')
        self.conv0 = nn.Conv2d(dim, dim, 5, padding=2, groups=dim)
        self.conv_spatial = nn.Conv2d(dim, dim, 7, stride=1, padding=9, groups=dim, dilation=3)
        self.conv1 = nn.Conv2d(dim, dim // 2, 1)
        self.conv2 = nn.Conv2d(dim, dim // 2, 1)
        self.conv_squeeze = nn.Conv2d(2, 2, 7, padding=3)
        self.conv = nn.Conv2d(dim // 2, dim, 1)

    def forward(self, x):
        attn1 = LF.DWConvFn.apply(x, self.conv0.weight, self.conv0.bias, 5, 1)
        attn2 = LF.DWConvFn.apply(attn1, self.conv_spatial.weight, self.conv_spatial.bias, 7, 3)
        attn1 = _conv1x1(self.conv1, attn1)
        attn2 = _conv1x1(self.conv2, attn2)
        attn = LF.LSKSelectFn.apply(attn1, attn2, self.conv_squeeze.weight, self.conv_squeeze.bias)
        attn = _conv1x1(self.conv, attn)
        return LF.MulFn.apply(x, attn)


class LKA(nn.Module):
    """VAN large-kernel attention (van_moe.py:319-333): x * conv1(conv_spatial(conv0(x)))."""

    def __init__(self, dim):
        super().__init__()
        if dim % 32:
            raise NotImplementedError(f'sm3det_b200: VAN width {dim} unsupported (multiple of 32)')
        self.conv0 = nn.Conv2d(dim, dim, 5, padding=2, groups=dim)
        self.conv_spatial = nn.Conv2d(dim, dim, 7, stride=1, padding=9, groups=dim, dilation=3)
        self.conv1 = nn.Conv2d(dim, dim, 1)

    def forward(self, x):
        attn = LF.DWConvFn.apply(x, self.conv0.weight, self.conv0.bias, 5, 1)
        attn = LF.DWConvFn.apply(attn, self.conv_spatial.weight, self.conv_spatial.bias, 7, 3)
        attn = _conv1x1(self.conv1, attn)
        return LF.MulFn.apply(x, attn)


class Attention(nn.Module):
    def __init__(self, d_model, unit='lsk'):
        super().__init__()
        self.proj_1 = nn.Conv2d(d_model, d_model, 1)
        self.activation = nn.GELU()
        self.spatial_gating_unit = LSKblock(d_model) if unit == 'lsk' else LKA(d_model)
        self.proj_2 = nn.Conv2d(d_model, d_model, 1)

    def forward(self, x):
        shortcut = x
        x = _conv1x1(self.proj_1, x, gelu=True)          # proj_1 + GELU fused in the GEMM epilogue
        x = self.spatial_gating_unit(x)
        x = _conv1x1(self.proj_2, x)
        return LF.AxpyFn.apply(x, shortcut, None, None)


class Block(nn.Module):
    def __init__(self, dim, mlp_ratio=4., drop=0., drop_path=0., act_layer=nn.GELU, norm_cfg=None, MoE_cfg1=None,
                 MoE_cfg2=None, unit='lsk'):
        super().__init__()
        self.norm1 = _build_bn(norm_cfg, dim)
        self.norm2 = _build_bn(norm_cfg, dim)
        self.attn = Attention(dim, unit)
        self.drop_path_rate = float(drop_path)
        self.drop_path = nn.Identity()
        self.MoE_cfg1, self.MoE_cfg2 = MoE_cfg1, MoE_cfg2
        self.mlp = Mlp(in_features=dim, hidden_features=int(dim * mlp_ratio), act_layer=act_layer, drop=drop,
                       MoE_cfg1=MoE_cfg1, MoE_cfg2=MoE_cfg2)
        layer_scale_init_value = 1e-2
        self.layer_scale_1 = nn.Parameter(layer_scale_init_value * torch.ones((dim)), requires_grad=True)
        self.layer_scale_2 = nn.Parameter(layer_scale_init_value * torch.ones((dim)), requires_grad=True)

    def forward(self, x, record=None):
        """x: NHWC.  Returns (x, loss or None)  (:387-396); both drop_path calls draw independent masks in the reference --
        an injected mask (tests) is shared by both, random masks are drawn twice."""
        rs1 = Fn.drop_path_row_scale(self, x)
        x = LF.AxpyFn.apply(self.attn(_bn(self.norm1, x)), x, self.layer_scale_1, rs1)
        rs2 = Fn.drop_path_row_scale(self, x)
        return self.mlp(_bn(self.norm2, x), self.layer_scale_2, x, rs2, record)


class OverlapPatchEmbed(nn.Module):
    def __init__(self, img_size=224, patch_size=7, stride=4, in_chans=3, embed_dim=768, norm_cfg=None):
        super().__init__()
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=stride,
                              padding=(patch_size // 2, patch_size // 2))
        self.norm = _build_bn(norm_cfg, embed_dim)

    def forward(self, x, nchw):
        x = LF.PatchEmbedFn.apply(x, self.proj.weight, self.proj.bias, self.proj.stride[0], nchw)
        return _bn(self.norm, x)


@ROTATED_BACKBONES.register_module()
class LSKNet_moe(BaseModule):
    _spatial_unit = 'lsk'          # 'lka' in the VAN subclasses (the only difference between lsk_moe.py and van_moe.py)

    def __init__(self, MoE_Block_inds_fc1=[[], [], [], []], MoE_Block_inds_fc2=[[], [], [], []], num_experts=2, top_k=2,
                 img_size=224, noisy_gating=False, gate='cosine', in_chans=3, embed_dims=[32, 64, 160, 256],
                 mlp_ratios=[8, 8, 4, 4], drop_rate=0., drop_path_rate=0., norm_layer=partial(nn.LayerNorm, eps=1e-6),
                 depths=[3, 3, 5, 2], num_stages=4, pretrained=None, init_cfg=None, norm_cfg=None):
        super().__init__(init_cfg=init_cfg)
        assert not (init_cfg and pretrained), 'init_cfg and pretrained cannot be set at the same time'
        if isinstance(pretrained, str):
            warnings.warn('DeprecationWarning: pretrained is deprecated, please use "init_cfg" instead')
            self.init_cfg = dict(type='Pretrained', checkpoint=pretrained)
        elif pretrained is not None:
            raise TypeError('pretrained must be a str or None')
        self.depths = depths
        self.embed_dims = embed_dims
        self.num_stages = num_stages
        self.num_experts = num_experts
        self.MoE_Block_inds_fc1 = MoE_Block_inds_fc1
        self.MoE_Block_inds_fc2 = MoE_Block_inds_fc2
        dpr = [x.item() for x in torch.linspace(0, drop_path_rate, sum(depths))]
        cur = 0
        for i in range(num_stages):
            depth = self.depths[i]
            ind1 = [list(range(depth))[q] for q in self.MoE_Block_inds_fc1[i] if q < depth]
            ind2 = [list(range(depth))[q] for q in self.MoE_Block_inds_fc2[i] if q < depth]
            patch_embed = OverlapPatchEmbed(img_size=img_size if i == 0 else img_size // (2 ** (i + 1)),
                                            patch_size=7 if i == 0 else 3, stride=4 if i == 0 else 2,
                                            in_chans=in_chans if i == 0 else embed_dims[i - 1], embed_dim=embed_dims[i],
                                            norm_cfg=norm_cfg)
            mk = lambda on: ({'noisy_gating': noisy_gating, 'num_experts': num_experts, 'top_k': top_k, 'gating': gate}
                             if on else None)
            block = nn.ModuleList([Block(dim=embed_dims[i], mlp_ratio=mlp_ratios[i], drop=drop_rate, drop_path=dpr[cur + j],
                                         norm_cfg=norm_cfg, MoE_cfg1=mk(j in ind1), MoE_cfg2=mk(j in ind2), unit=self._spatial_unit)
                                   for j in range(depths[i])])
            norm = norm_layer(embed_dims[i])
            cur += depths[i]
            setattr(self, f'patch_embed{i + 1}', patch_embed)
            setattr(self, f'block{i + 1}', block)
            setattr(self, f'norm{i + 1}', norm)

    # ---- checkpoint up-cycling (lsk_moe.py:473-523): dense fc1/fc2 weights copied into every expert ----------
    def upcycle_state_dict(self, src):
        out = {}
        for k, v in src.items():
            if k.startswith('head'):
                continue
            if k.startswith('block') and 'fc' in k:
                parts = k[5:].split('.')
                stage_ind, block_ind = int(parts[0]) - 1, int(parts[1])
                which = 'fc1' if 'fc1' in k else 'fc2'
                inds = self.MoE_Block_inds_fc1 if which == 'fc1' else self.MoE_Block_inds_fc2
                if block_ind in inds[stage_ind]:
                    for e in range(self.num_experts):
                        out[k.replace(which, f'{which}.experts.{e}')] = v
                else:
                    out[k] = v
            else:
                out[k] = v
        return out

    def init_weights(self):
        """lsk_moe.py:473-523 / :766-826: init_cfg=None -> from-scratch initialisation (Linear trunc-normal 0.02,
        LayerNorm (1, 0), Conv2d fan-out normal); a Pretrained dict -> up-cycle the dense checkpoint."""
        cfg = self.init_cfg
        if cfg is None:
            for m in self.modules():
                if isinstance(m, nn.Linear):
                    nn.init.trunc_normal_(m.weight, mean=0., std=.02, a=-2., b=2.)
                    if m.bias is not None:
                        nn.init.constant_(m.bias, 0.)
                elif isinstance(m, nn.LayerNorm):
                    nn.init.constant_(m.weight, 1.0)
                    nn.init.constant_(m.bias, 0.)
                elif isinstance(m, nn.Conv2d):
                    fan_out = m.kernel_size[0] * m.kernel_size[1] * m.out_channels // m.groups
                    nn.init.normal_(m.weight, 0., math.sqrt(2.0 / fan_out))
                    if m.bias is not None:
                        nn.init.constant_(m.bias, 0.)
            return
        if isinstance(cfg, dict) and cfg.get('type') == 'Pretrained' and cfg.get('checkpoint'):
            ckpt = torch.load(cfg['checkpoint'], map_location='cpu')
            sd = ckpt.get('state_dict', ckpt.get('model', ckpt))
            print(self.load_state_dict(self.upcycle_state_dict(sd), strict=False))

    def freeze_patch_emb(self):
        self.patch_embed1.requires_grad = False

    @staticmethod
    def _check_input(x):
        if not x.is_cuda:
            raise RuntimeError('sm3det_b200 backbones run on CUDA (sm_100a) only; there is no CPU path')
        if x.dim() != 4:
            raise ValueError(f'expected [N,C,H,W], got {tuple(x.shape)}')

    def _stage_tail(self, i, x, outs, gate_losses, record):
        for blk in getattr(self, f'block{i + 1}'):
            x, gate_loss = blk(x, record)
            if gate_loss is not None:
                gate_losses.append(gate_loss)
        nl = getattr(self, f'norm{i + 1}')
        # LayerNorm over C + NHWC->NCHW (:555-557); the NORMED map is both the returned feature and the next stage's input
        outs.append(Fn.OutNormFn.apply(x, nl.weight, nl.bias, nl.eps))
        return outs[-1]

    def forward_features(self, x, record=None):
        outs, gate_losses = [], []
        for i in range(self.num_stages):
            x = getattr(self, f'patch_embed{i + 1}')(x, nchw=True)
            x = self._stage_tail(i, x, outs, gate_losses, record)
        if len(gate_losses) > 0:
            return tuple(outs), sum(gate_losses) / len(gate_losses)
        return tuple(outs)

    def _precision(self):
        from . import ops
        return ops.precision_scope(ops.autocast_passes(self))     # scoped to this call (see ops.captures_precision)

    def forward(self, x, record=None):
        self._check_input(x)
        with self._precision():
            return self.forward_features(x, record)


@ROTATED_BACKBONES.register_module()
class LSKNet_moe_MultiInput(LSKNet_moe):
    def __init__(self, in_channels=3, datasets=None, inject_uni_info_mode=None, norm_cfg=None, drop_path_rate=0.,
                 MoE_Block_inds_fc1=[[], [], [], []], MoE_Block_inds_fc2=[[], [], [], []], noisy_gating=True, num_experts=2,
                 gate='cosine', top_k=2,
                 init_cfg=[dict(type='TruncNormal', layer=['Conv2d', 'Linear'], std=.02, bias=0.),
                           dict(type='Constant', layer=['LayerNorm'], val=1., bias=0.)],
                 img_size=256, embed_dims=[32, 64, 160, 256], mlp_ratios=[8, 8, 4, 4], drop_rate=0.,
                 norm_layer=partial(nn.LayerNorm, eps=1e-6), depths=[3, 3, 5, 2], num_stages=4, pretrained=None):
        super().__init__(MoE_Block_inds_fc1=MoE_Block_inds_fc1, MoE_Block_inds_fc2=MoE_Block_inds_fc2,
                         num_experts=num_experts, top_k=top_k, img_size=img_size, noisy_gating=noisy_gating, gate=gate,
                         in_chans=in_channels, embed_dims=embed_dims, mlp_ratios=mlp_ratios, drop_rate=drop_rate,
                         drop_path_rate=drop_path_rate, norm_layer=norm_layer, depths=depths, num_stages=num_stages,
                         pretrained=pretrained, init_cfg=init_cfg, norm_cfg=norm_cfg)
        if datasets is not None or inject_uni_info_mode is not None:
            raise NotImplementedError('sm3det_b200: per-dataset stems / inject_uni_info_mode are not implemented '
                                      '(every SM3Det config uses datasets=None)')
        self.init_datasets = datasets
        self.datasets = ['single']
        self.inject_uni_info_mode = inject_uni_info_mode
        self.use_uni_head = False
        self.dataset_stems = nn.ModuleDict()
        for dataset in self.datasets:
            self.dataset_stems[dataset] = self.patch_embed1.proj
        self.patch_embed1 = _build_bn(norm_cfg, embed_dims[0])          # patch_embed1 becomes the BN only (:692-695)

    def upcycle_state_dict(self, src):
        """lsk_moe.py:806-813: on top of the expert remap, the dense checkpoint's stem conv 'patch_embed1.proj.*' moves to
        'dataset_stems.single.*' and its BatchNorm 'patch_embed1.norm.*' to 'patch_embed1.*' (patch_embed1 is the BN only)."""
        out = {}
        for k, v in super().upcycle_state_dict(src).items():
            if k.startswith('patch_embed1'):
                if 'norm' in k:
                    out[k.replace('.norm.', '.')] = v
                else:
                    for d in self.datasets:
                        out[k.replace('patch_embed1.proj', 'dataset_stems.' + str(d))] = v
            else:
                out[k] = v
        return out

    def forward_features(self, x, record=None):
        outs, gate_losses = [], []
        for i in range(self.num_stages):
            pe = getattr(self, f'patch_embed{i + 1}')
            x = _bn(pe, x) if i == 0 else pe(x, nchw=True)
            x = self._stage_tail(i, x, outs, gate_losses, record)
        if len(gate_losses) > 0:
            return tuple(outs), sum(gate_losses) / len(gate_losses)
        return tuple(outs)

    def forward(self, x, datasets=['single'], record=None):
        if len(datasets) == 1:
            x = [x]
        x = torch.cat(list(x), dim=0)                                   # one shared stem (:751-754)
        self._check_input(x)
        with self._precision():
            stem = self.dataset_stems['single']
            x = LF.PatchEmbedFn.apply(x, stem.weight, stem.bias, stem.stride[0], True)
            return self.forward_features(x, record)


@ROTATED_BACKBONES.register_module()
class VAN_moe(LSKNet_moe):
    """van_moe.py:410-588: identical to LSKNet_moe except the spatial gating unit (LKA, :319-333)."""
    _spatial_unit = 'lka'


@ROTATED_BACKBONES.register_module()
class VAN_moe_MultiInput(LSKNet_moe_MultiInput):
    """van_moe.py:590-814."""
    _spatial_unit = 'lka'
