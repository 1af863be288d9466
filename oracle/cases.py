"""Golden-case definitions shared by oracle/gen_golden.py and the tests (test infrastructure)."""
import contextlib

import torch

# torch's CPU convolutions split their reductions by the number of intra-op threads, so the oracle reproduces the fixtures
# bit-for-bit only at the thread count they were generated with
GOLDEN_THREADS = 8


@contextlib.contextmanager
def golden_threads():
    """Run torch's CPU ops with the thread count the fixtures were generated with."""
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(n)


MINI = dict(depths=[1, 1, 2, 1], channels=[32, 64, 96, 128])
MINI2 = dict(depths=[2, 2, 3, 2], channels=[32, 64, 128, 256])

# name -> (constructor kwargs, image spec, mode)
CASES = {
    # BASELINE config 1: ConvNeXt-T, no MoE, 1x3x256x256, eval forward
    'tiny_dense_256': dict(kw=dict(arch='tiny'), img=(1, 256, 256), mode='eval', weights='trained', stride=4),
    'tiny_dense_256_init': dict(kw=dict(arch='tiny'), img=(1, 256, 256), mode='eval', weights='init', stride=4),
    'mini_dense': dict(kw=dict(arch=MINI), img=(2, 64, 64), mode='eval', weights='trained', stride=1),
    'mini_moe_e4k2_eval': dict(kw=dict(arch=MINI, MoE_Block_inds=[[], [0], [0, 1], [0]], num_experts=4, top_k=2),
                               img=(2, 64, 96), mode='eval', weights='trained', stride=1),
    'mini_moe_e8k3_eval': dict(kw=dict(arch=MINI, MoE_Block_inds=[[0], [0], [1], [0]], num_experts=8, top_k=3),
                               img=(3, 64, 64), mode='eval', weights='trained', stride=1),
    'mini_moe_e6k1_eval': dict(kw=dict(arch=MINI, MoE_Block_inds=[[], [], [0, 1], []], num_experts=6, top_k=1),
                               img=(2, 96, 64), mode='eval', weights='trained', stride=1),
    'mini_moe_e2k2_eval': dict(kw=dict(arch=MINI, MoE_Block_inds=[[], [], [0], [0]], num_experts=2, top_k=2),
                               img=(2, 64, 64), mode='eval', weights='trained', stride=1),
    'mini_moe_e4k2_train_clean': dict(kw=dict(arch=MINI, MoE_Block_inds=[[], [0], [0, 1], [0]], num_experts=4, top_k=2,
                                              noisy_gating=False),
                                      img=(2, 64, 64), mode='train', weights='trained', stride=1),
    'mini_moe_e4k2_train_noisy': dict(kw=dict(arch=MINI, MoE_Block_inds=[[], [0], [0, 1], [0]], num_experts=4, top_k=2),
                                      img=(2, 64, 64), mode='train_noisy', weights='trained', stride=1),
    'mini2_moe_e8k2_train_clean': dict(kw=dict(arch=MINI2, MoE_Block_inds=[[], [], [0, 2], [0]], num_experts=8, top_k=2,
                                               noisy_gating=False),
                                       img=(2, 128, 128), mode='train', weights='trained', stride=2),
}

# ---- ConvNeXt_DA_MultiInput (convnext_moe_DA.py, local_configs/main_DA_convnext_t_orcnn_gfl.py): a DALayer per block ----
# `datasets`: one name = whole batch through that dataset's gate; three names = one image per modality (the detector's call)
DA_CASES = {
    'da_mini_dense_eval_rgb': dict(kw=dict(arch=MINI), img=(2, 64, 64), mode='eval', weights='trained', stride=1, da=True,
                                   datasets=['rgb']),
    'da_mini_dense_train_3mod': dict(kw=dict(arch=MINI), img=(3, 64, 64), mode='train', weights='trained', stride=1, da=True,
                                     datasets=['sar', 'rgb', 'ifr']),
    'da_mini_moe_e4k2_train_noisy_3mod': dict(kw=dict(arch=MINI, MoE_Block_inds=[[], [0], [0, 1], [0]], num_experts=4, top_k=2),
                                              img=(3, 64, 96), mode='train_noisy', weights='trained', stride=1, da=True,
                                              datasets=['sar', 'rgb', 'ifr']),
}
CASES.update(DA_CASES)

# ---- full-size cases: the shapes bench.py times (BASELINE configs 2/3, the shipped k=3 recipe, config 4's widths) -----
# One 1024^2 (or 512^2) image each; fixtures keep strided output samples, compact routing (int8 indices + the oracle's own
# (k)-vs-(k+1) logit gap per token, which is what decides whether a routing flip is a numerical tie) and gradient digests.
CFG2_KW = dict(arch='tiny', MoE_Block_inds=[[], [], [0, 2, 4, 6, 8], [0, 2]], num_experts=8, top_k=2)
CFG4_KW = dict(arch='base', MoE_Block_inds=[[0, 1, 2], [0, 1, 2], list(range(27)), [0, 1, 2]], num_experts=16, top_k=2)
FULL_CASES = {
    'cfg2_t_e8k2_1024_eval': dict(kw=dict(CFG2_KW), img=(1, 1024, 1024), mode='eval', weights='trained', stride=8),
    'cfg2_t_e8k2_1024_train_clean': dict(kw=dict(CFG2_KW, noisy_gating=False), img=(1, 1024, 1024), mode='train',
                                         weights='trained', stride=8),
    'cfg2_t_e8k2_1024_train_noisy': dict(kw=dict(CFG2_KW), img=(1, 1024, 1024), mode='train_noisy', weights='trained',
                                         stride=8),
    # configs/SM3Det/SM3Det_convnext_t.py:15-19 (shipped recipe: top_k = 3)
    'ship_t_e8k3_512_train_noisy': dict(kw=dict(CFG2_KW, top_k=3), img=(2, 512, 512), mode='train_noisy', weights='trained',
                                        stride=4),
    # BASELINE config 4: ConvNeXt-B, E = 16, all 36 blocks MoE (C = 128 / 256 / 512 / 1024)
    'cfg4_b_e16k2_512_train_clean': dict(kw=dict(CFG4_KW, noisy_gating=False), img=(1, 512, 512), mode='train',
                                         weights='trained', stride=4),
}
for _v in FULL_CASES.values():
    _v['full'] = True
CASES.update(FULL_CASES)


def upstream_grads(outs, seed=99):
    """Seeded upstream gradients for the 4 outputs (SURVEY.md 8d): randn / sqrt(numel)."""
    gs = []
    for i, o in enumerate(outs):
        g = torch.Generator().manual_seed(seed + i)
        gs.append(torch.randn(o.shape, generator=g) / (o.numel() ** 0.5))
    return gs


def make_noise(cfg, n_tokens_per_layer, seed=7):
    out = []
    for i, t in enumerate(n_tokens_per_layer):
        g = torch.Generator().manual_seed(seed + i)
        out.append(torch.randn(t, cfg.num_experts, generator=g))
    return out


def summarize_grad(g: torch.Tensor, full_below=4096, samples=256):
    g = g.detach().float().reshape(-1)
    if g.numel() <= full_below:
        return dict(full=g.clone())
    idx = torch.linspace(0, g.numel() - 1, samples).long()
    return dict(sample=g[idx].clone(), idx=idx, l2=g.double().norm().item(), s=g.double().sum().item())


def assert_matches_summary(t: torch.Tensor, s: dict, what=''):
    """t reproduces the tensor summarize_grad summarised as s bit-for-bit: every stored element equal, the full tensor's
    float64 L2 norm and sum equal up to the summation order of the CPU kernels."""
    t = t.detach().float().reshape(-1)
    if 'full' in s:
        assert torch.equal(t, s['full']), f'{what}: differs by {(t - s["full"]).abs().max()}'
        return
    assert torch.equal(t[s['idx']], s['sample']), f'{what}: sampled elements differ by {(t[s["idx"]] - s["sample"]).abs().max()}'
    assert abs(t.double().norm().item() - s['l2']) <= 1e-12 * s['l2'], what
    assert abs(t.double().sum().item() - s['s']) <= 1e-12 * s['l2'] * t.numel() ** 0.5, what


# ---- LSKNet-MoE (BASELINE config 5 family; oracle/lsk_moe_oracle.py) --------------------------------------------
LSK_MINI = dict(embed_dims=[64, 64, 128, 128], depths=[1, 1, 2, 1], mlp_ratios=[4, 4, 2, 2])
LSK_CASES = {
    'lsk_mini_dense_eval': dict(kw=dict(**LSK_MINI), img=(2, 64, 64), mode='eval'),
    'lsk_mini_moe_e4k2_eval': dict(kw=dict(**LSK_MINI, MoE_Block_inds_fc1=[[], [0], [0, 1], [0]],
                                           MoE_Block_inds_fc2=[[], [0], [0, 1], [0]], num_experts=4, top_k=2),
                               img=(2, 64, 96), mode='eval'),
    'lsk_mini_moe_e4k2_train_clean': dict(kw=dict(**LSK_MINI, MoE_Block_inds_fc1=[[0], [0], [0, 1], [0]],
                                                  MoE_Block_inds_fc2=[[], [0], [1], [0]], num_experts=4, top_k=2,
                                                  noisy_gating=False),
                                      img=(2, 64, 64), mode='train'),
    'lsk_mini_moe_e3k1_train_noisy_drop': dict(kw=dict(**LSK_MINI, MoE_Block_inds_fc1=[[], [0], [0], [0]],
                                                       MoE_Block_inds_fc2=[[], [0], [0, 1], []], num_experts=3, top_k=1,
                                                       drop_rate=0.1),
                                           img=(3, 64, 64), mode='train_noisy'),
}

# BASELINE config 5 at its real widths (configs/SM3Det/SM3Det_lsk_s.py:14-25).  Batch 2, not 1: at batch size 1 torch 2.11's
# CPU autograd returns gradients for this op sequence that disagree with finite differences of its own forward (the
# unmodified reference and the oracle alike -- tests/diag/fd_check_lsk_oracle.py), so batch-1 gradient fixtures would pin a
# framework artefact.  Forward outputs are unaffected.
LSK_S_KW = dict(embed_dims=[64, 128, 320, 512], depths=[2, 2, 4, 2], MoE_Block_inds_fc1=[[], [0], [0, 2], [0]],
                MoE_Block_inds_fc2=[[], [0], [0, 2], [0]], num_experts=4, top_k=2)
LSK_CASES.update({
    'lsk_s_cfg5_1024_eval': dict(kw=dict(LSK_S_KW), img=(1, 1024, 1024), mode='eval', full=True, stride=8),
    'lsk_s_cfg5_b2_768_train_noisy_drop': dict(kw=dict(LSK_S_KW, drop_rate=0.1), img=(2, 768, 768), mode='train_noisy',
                                               full=True, stride=8),
})

VAN_MINI = dict(embed_dims=[32, 64, 96, 128], depths=[1, 1, 2, 1], mlp_ratios=[4, 4, 2, 2])
LSK_CASES.update({
    # VAN-MoE (van_moe.py = lsk_moe.py with the LKA gating unit); fixtures are named van_*.pt
    'van_mini_moe_e4k2_eval': dict(kw=dict(**VAN_MINI, MoE_Block_inds_fc1=[[], [0], [0, 1], [0]],
                                           MoE_Block_inds_fc2=[[0], [0], [1], [0]], num_experts=4, top_k=2),
                               img=(2, 64, 64), mode='eval', unit='lka'),
    'van_mini_moe_e4k2_train_noisy': dict(kw=dict(**VAN_MINI, MoE_Block_inds_fc1=[[], [0], [0, 1], [0]],
                                                  MoE_Block_inds_fc2=[[0], [0], [1], []], num_experts=4, top_k=2),
                                      img=(2, 64, 64), mode='train_noisy', unit='lka'),
})


def lsk_plan(cfg, n, h, w):
    """Per MoE layer (in forward order) its token count, and per dropout call its tensor shape [N,C,H,W]."""
    tokens, drops = [], []
    for i in range(cfg.num_stages):
        hh, ww = h // (4 * 2 ** i), w // (4 * 2 ** i)
        hid = int(cfg.embed_dims[i] * cfg.mlp_ratios[i])
        for j in range(cfg.depths[i]):
            if j in cfg.moe_fc1(i):
                tokens.append(n * hh * ww)
            if j in cfg.moe_fc2(i):
                tokens.append(n * hh * ww)
            drops.append((n, hid, hh, ww))
            drops.append((n, cfg.embed_dims[i], hh, ww))
    return tokens, drops


def make_drop_masks(shapes, rate, seed=31):
    out = []
    for i, s in enumerate(shapes):
        g = torch.Generator().manual_seed(seed + i)
        out.append((torch.rand(s, generator=g) >= rate).float() / (1.0 - rate))
    return out


def lsk_injections(cfg, gold):
    """(noise list, dropout mask list) a fixture's training mode injects, in forward order (None when inactive)."""
    n, h, w = gold['img']
    tokens, dshapes = lsk_plan(cfg, n, h, w)
    noise = drops = None
    if gold['mode'] == 'train_noisy':
        noise = [torch.randn(t, cfg.num_experts, generator=torch.Generator().manual_seed(7 + i)) for i, t in enumerate(tokens)]
    if cfg.drop_rate > 0 and gold['mode'] != 'eval':
        drops = make_drop_masks(dshapes, cfg.drop_rate)
    return noise, drops
