"""N-GPU worker: expert-parallel MoE ConvNeXt backbone (NVLink peer gathers) vs the same backbone with all experts local,
with clean and with noisy gating.  Launched by tests/test_ep_gpu.py through torch.distributed.run (one process per GPU,
NCCL)."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, sys.argv[1])
from oracle.cases import make_noise  # noqa: E402
from oracle.convnext_moe_oracle import OracleConfig, param_shapes  # noqa: E402  (shapes only)
from oracle.gen_golden import moe_token_counts  # noqa: E402
from sm3det_b200 import ConvNeXt_moe_MultiInput  # noqa: E402
from sm3det_b200.expert_parallel import enable_expert_parallel  # noqa: E402
from sm3det_b200.synth import make_images, make_state_dict  # noqa: E402


def rel(a, b):
    return ((a - b).abs().max() / (b.abs().max() + 1e-30)).item()


def compare(rank, W, ep_group, noisy):
    kw = dict(arch=dict(depths=[1, 1, 2, 1], channels=[32, 64, 96, 128]), MoE_Block_inds=[[], [0], [0, 1], [0]],
              num_experts=2 * W, top_k=2, noisy_gating=noisy)
    cfg = OracleConfig(**kw)
    sd = make_state_dict(param_shapes(cfg), 0, True)
    # the same seeded gating noise for both nets (its own draw on every rank, like the images)
    noise = make_noise(cfg, moe_token_counts(cfg, 2, 64, 64), seed=7 + 100 * rank) if noisy else None
    nets = []
    for _ in range(2):
        net = ConvNeXt_moe_MultiInput(**kw)
        net.load_state_dict(sd, strict=True)
        if noisy:
            for m, nz in zip([m for m in net.modules() if m.__class__.__name__ == 'MoE_layer'], noise, strict=True):
                m._injected_noise = nz
        nets.append(net.cuda().train())
    ref, epn = nets
    assert enable_expert_parallel(epn, ep_group, average_grads=False) == 4
    x = make_images(2, 64, 64, seed=500 + rank).cuda()            # different images on every rank
    outs_r, loss_r = ref(x)
    outs_e, loss_e = epn(x)
    fe = max(rel(a, b) for a, b in zip(outs_e, outs_r))
    assert fe < 1e-5, f'rank {rank}: EP forward differs from the local-experts forward by {fe}'
    assert abs(loss_e.item() - loss_r.item()) <= 1e-6 * abs(loss_r.item()) + 1e-9
    ups = [torch.randn(o.shape, generator=torch.Generator().manual_seed(7 + i + 10 * rank)).cuda() / o.numel() ** 0.5
           for i, o in enumerate(outs_r)]
    (sum((o * g).sum() for o, g in zip(outs_r, ups)) + loss_r).backward()
    (sum((o * g).sum() for o, g in zip(outs_e, ups)) + loss_e).backward()
    torch.cuda.synchronize()
    epn._ep_ctx.check()                                        # no capacity overflow
    El = 2
    worst = 0.0
    for (n, pr), (_, pe) in zip(ref.named_parameters(), epn.named_parameters()):
        gr, ge = pr.grad, pe.grad
        if '.experts.' in n:
            e = int(n.split('.experts.')[1].split('.')[0])
            tot = gr.clone()
            dist.all_reduce(tot)                               # expert e saw tokens of every rank on its owner
            if e // El == rank:
                err = rel(ge, tot)
            else:
                assert ge is None, n                           # not owned: no gradient at all (stays out of the DDP buckets)
                continue
        else:
            err = rel(ge, gr)
        worst = max(worst, err)
        assert err < 2e-4, f'rank {rank}: grad {n} differs by {err}'
        if n.endswith('.w_noise'):
            assert bool(gr.abs().max() > 0) == noisy, f'rank {rank}: {n} gradient {float(gr.abs().max())} (noisy={noisy})'
    print(f'rank {rank}: ep ok noisy={noisy} fwd {fe:.2e} worst grad {worst:.2e}')


def main():
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dist.init_process_group('nccl')
    rank, W = dist.get_rank(), dist.get_world_size()
    ep_group = dist.new_group(list(range(W)))
    for noisy in (False, True):
        compare(rank, W, ep_group, noisy)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
