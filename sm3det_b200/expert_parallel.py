"""Expert-parallel MoE block over NVLink peer memory (BASELINE config 4; beyond the reference, SURVEY.md 8e).

The reference runs every expert on every rank (DDP).  Here the E experts of a layer are partitioned over the W ranks of
one NVSwitch box (rank d owns experts [d*E/W, (d+1)*E/W)); tokens stay where they are and the two "all-to-all" steps of
SparseDispatcher (dispatch :264-266, combine :269-284 of convnext_moe.py) become *direct NVLink loads*:

  dispatch : the expert rank gathers the rows routed to its experts straight out of the source ranks' LayerNorm output
             (sm3_gather_rows_peer through the source's expert-sorted pair list) -- no send buffer, no NCCL on the data path;
  combine  : the source rank gathers its pairs' expert outputs straight out of the expert ranks' output buffers and runs
             the same deterministic moe_combine kernel as the single-GPU path.
  backward : mirrors it (d_o rows pulled by the expert rank, d_x rows pulled back by the source rank).

Only two tiny collectives per layer and direction remain: an all_gather of the [2,E] count / segment table (which also
orders "LayerNorm output written" before "peers read it") and a 1-element all_reduce used as a stream-ordered barrier.
The exchange plan is built on the device from that table (sm3_ep_plan) -- there is NO host synchronisation per layer; the
expert-side row space has a fixed capacity (capacity_factor x the balanced load, 2x by default) and an overflow is reported
by a device flag that `EPContext.check()` reads off the critical path.
Buffers that peers read live in torch symmetric memory (CUDA P2P mappings); every kernel is launched on the current
stream.  Expert parameters keep the reference's names and shapes on every rank (state_dict compatible); a rank only ever
touches -- and produces non-zero gradients for -- the experts it owns, so wrapping the model in DDP (mean over ranks)
yields exactly the data-parallel gradient.  Expert parameters are meant to stay OUT of the DDP buckets
(`ddp_ignored_parameters`): a rank produces gradients only for the experts it owns (already scaled by 1/world, i.e. DDP's
mean) and None for the others, so nothing expert-sized is ever all-reduced.
"""
import torch
import torch.distributed as dist
from torch.autograd import Function

from . import functional as Fn
from . import ops


class EPContext:
    """Process-wide expert-parallel state: group, symmetric buffers (shared by all layers of one shape) and their peer
    pointer tables."""

    def __init__(self, group=None, capacity_factor=2.0, average_grads=True):
        self.group = group if group is not None else dist.group.WORLD
        self.world = dist.get_world_size(self.group)
        self.rank = dist.get_rank(self.group)
        self.capacity_factor = capacity_factor      # None = worst case (every pair of every rank lands on one rank)
        self.average_grads = average_grads          # scale owned-expert gradients by 1/world (what DDP's mean would do)
        self._bufs = {}
        self._flag = None
        self.overflow = None

    # -- symmetric memory -------------------------------------------------------------------------------------
    def _symm(self, numel, dtype):
        import torch.distributed._symmetric_memory as symm_mem
        t = symm_mem.empty(numel, dtype=dtype, device=torch.device('cuda', torch.cuda.current_device()))
        try:
            hdl = symm_mem.rendezvous(t, self.group)
        except TypeError:
            hdl = symm_mem.rendezvous(t, self.group.group_name)
        ptrs = torch.tensor([int(p) for p in hdl.buffer_ptrs], dtype=torch.int64, device=t.device)
        return t, ptrs, hdl

    def buffers(self, T, C, k, E):
        """Symmetric buffers for MoE layers with T local tokens of width C, allocated (collectively) on first use and
        shared by every layer of that shape: the per-layer collectives order one layer's peer reads before the next
        layer's writes.  All ranks must present the same T (identical N*H*W per rank) -- checked here, once."""
        key = (T, C, k, E)
        b = self._bufs.get(key)
        if b is not None:
            return b
        W = self.world
        t = torch.tensor([T, -T], device='cuda', dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        if int(t[0]) != T or int(t[1]) != -T:
            raise RuntimeError(f'sm3det_b200 expert parallelism needs the same number of tokens (N*H*W) on every rank; this rank '
                               f'has {T}, the group spans {-int(t[1])}..{int(t[0])}')
        R_s = ((T * k + 127) // 128 + E) * 128                       # padded local slot space (moe_plan)
        pairs = W * T * k if self.capacity_factor is None else min(W * T * k, int(self.capacity_factor * T * k))
        cap = ((pairs + 127) // 128 + E // W) * 128                  # padded expert-side row space
        b = dict(T=T, R_s=R_s, cap=cap)
        b['v'], b['v_ptrs'], _ = self._symm(T * C, torch.float32)
        b['pair'], b['pair_ptrs'], _ = self._symm(R_s, torch.int32)
        b['o'], b['o_ptrs'], _ = self._symm(cap * C, torch.float32)
        b['do'], b['do_ptrs'], _ = self._symm(R_s * C, torch.float32)
        b['dxp'], b['dxp_ptrs'], _ = self._symm(cap * C, torch.float32)
        self._bufs[key] = b
        if self.overflow is None:
            self.overflow = torch.zeros(1, device='cuda', dtype=torch.int32)
        return b

    def barrier(self):
        """Stream-ordered cross-rank barrier (1-element NCCL all_reduce on the current stream)."""
        if self._flag is None:
            self._flag = torch.zeros(1, device='cuda')
        dist.all_reduce(self._flag, group=self.group)

    def check(self):
        """Raise if any layer's expert-side rows ever exceeded the capacity (synchronises: call it off the critical path)."""
        if self.overflow is not None and int(self.overflow) > 0:
            raise RuntimeError(f'sm3det_b200: expert-parallel capacity exceeded ({int(self.overflow)} rows needed); '
                               f'raise capacity_factor (now {self.capacity_factor})')


def device_plan(ctx, allm, tile_group_s, num_tiles_s, pair_token, E, R_s, cap):
    """sm3_ep_plan: the exchange plan of one layer, entirely on the device (same content as _build_plan, capacity-bounded)."""
    import ctypes as C
    from . import _lib
    dev = pair_token.device
    El = E // ctx.world
    i = torch.empty(2 * cap + cap // 128 + 1 + 2 * El + 2 * R_s, device=dev, dtype=torch.int32)
    o = 0

    def take(n):
        nonlocal o
        t = i[o:o + n]
        o += n
        return t
    P = dict(cap=cap, src_rank=take(cap), src_slot=take(cap), tile_group=take(cap // 128), num_tiles=take(1),
             seg_begin=take(El), seg_end=take(El), comb_rank=take(R_s), comb_row=take(R_s))
    a = _lib.EpPlanArgs()
    a.allm = allm.data_ptr(); a.tile_group_s = tile_group_s.data_ptr(); a.num_tiles_s = num_tiles_s.data_ptr()
    a.pair_token = pair_token.data_ptr()
    a.W, a.me, a.E, a.R_s, a.cap = ctx.world, ctx.rank, E, R_s, cap
    for name in ('src_rank', 'src_slot', 'tile_group', 'num_tiles', 'seg_begin', 'seg_end', 'comb_rank', 'comb_row'):
        setattr(a, name, P[name].data_ptr())
    a.overflow = ctx.overflow.data_ptr()
    _lib.check(_lib.load().sm3_ep_plan(C.byref(a), torch.cuda.current_stream().cuda_stream), 'sm3_ep_plan')
    return P


def _expert_layout(cnt, W, E):
    """Host-side plan from the gathered counts cnt[W,E] (python ints): for every owner rank d the padded start of each of
    its experts and, per (expert, source) block, the row offset.  Identical on all ranks."""
    E_loc = E // W
    seg = [[0] * E_loc for _ in range(W)]        # seg[d][e_loc]  first row of the expert on its owner
    off = [[0] * W for _ in range(E)]            # off[g][s]      offset of source s inside expert g's segment
    rows = [0] * W                               # padded row count per owner
    tiles = [[] for _ in range(W)]               # tile -> local expert id, per owner
    for d in range(W):
        pos = 0
        for el in range(E_loc):
            g = d * E_loc + el
            seg[d][el] = pos
            acc = 0
            for s in range(W):
                off[g][s] = acc
                acc += cnt[s][g]
            nt = (acc + 127) // 128
            tiles[d] += [el] * nt
            pos += nt * 128
        rows[d] = pos
    return seg, off, rows, tiles


def _build_plan(ctx, cnt_all, seg_all, tile_group_s, num_tiles_s, pair_token, E, R_s, dev):
    """Index tensors of one layer (plumbing on small / index-only tensors; no activation arithmetic)."""
    W, me = ctx.world, ctx.rank
    E_loc = E // W
    cnt = cnt_all.tolist()                                   # host sync (the reference syncs twice per layer, :254,:259)
    segs = seg_all.tolist()
    seg, off, rows, tiles = _expert_layout(cnt, W, E)
    R_d = rows[me]
    # ---- expert side: row r of my padded expert-major space <- (source rank, slot in that rank's pair list)
    L, D, S, SR = [], [], [], []
    for el in range(E_loc):
        g = me * E_loc + el
        for s in range(W):
            if cnt[s][g] > 0:
                L.append(cnt[s][g]); D.append(seg[me][el] + off[g][s]); S.append(segs[s][g]); SR.append(s)
    src_rank = torch.full((max(R_d, 1),), -1, device=dev, dtype=torch.int32)
    src_slot = torch.zeros((max(R_d, 1),), device=dev, dtype=torch.int32)
    if L:
        Lt = torch.tensor(L, device=dev)
        blk = torch.repeat_interleave(torch.arange(len(L), device=dev), Lt)
        within = torch.arange(int(Lt.sum()), device=dev) - torch.repeat_interleave(torch.cumsum(Lt, 0) - Lt, Lt)
        dest = torch.tensor(D, device=dev)[blk] + within
        src_rank[dest] = torch.tensor(SR, device=dev, dtype=torch.int32)[blk]
        src_slot[dest] = (torch.tensor(S, device=dev)[blk] + within).to(torch.int32)
    seg_b = [seg[me][el] for el in range(E_loc)]
    seg_e = [seg[me][el] + sum(cnt[s][me * E_loc + el] for s in range(W)) for el in range(E_loc)]
    plan = dict(R_d=R_d, src_rank=src_rank, src_slot=src_slot,
                tile_group=torch.tensor(tiles[me] + [0], device=dev, dtype=torch.int32),
                num_tiles=torch.tensor([len(tiles[me])], device=dev, dtype=torch.int32),
                seg_begin=torch.tensor(seg_b, device=dev, dtype=torch.int32),
                seg_end=torch.tensor(seg_e, device=dev, dtype=torch.int32))
    # ---- source side: my slot l (expert g) lives on rank g // E_loc at row  l - seg_s[g] + seg[owner][e_loc] + off[g][me]
    delta = torch.tensor([seg[g // E_loc][g % E_loc] + off[g][me] - segs[me][g] for g in range(E)], device=dev)
    owner = torch.tensor([g // E_loc for g in range(E)], device=dev, dtype=torch.int32)
    g_of_slot = torch.repeat_interleave(tile_group_s[:R_s // 128].long().clamp_(0, E - 1), 128)
    slot = torch.arange(R_s, device=dev)
    live = (slot < num_tiles_s.long() * 128) & (pair_token >= 0)
    plan['comb_rank'] = torch.where(live, owner[g_of_slot], torch.full_like(owner[g_of_slot], -1)).contiguous()
    plan['comb_row'] = torch.where(live, slot + delta[g_of_slot], torch.zeros_like(slot)).to(torch.int32).contiguous()
    return plan


@ops.captures_precision
class EPMoEBlockFn(Function):
    """ConvNeXt MoE block with expert-parallel experts: dwconv -> LN -> router (local) -> P2P dispatch -> owned experts ->
    P2P combine (+ gamma + shortcut).  Same math as functional.MoEBlockFn; experts[...] are ALL E experts' parameters."""

    @staticmethod
    def forward(ctx, x, dww, dwb, lnw, lnb, gamma, wp, bp, sim, tau, w_noise, row_scale, noise, eps, E, k, record, packs, ep,
                key, *experts):
        N, H, W_, C = x.shape
        T = N * H * W_
        Wn, me = ep.world, ep.rank
        assert E % Wn == 0, 'expert parallelism needs num_experts divisible by the world size'
        E_loc = E // Wn
        w1s, b1s, w2s, b2s = experts[0:E], experts[E:2 * E], experts[2 * E:3 * E], experts[3 * E:4 * E]
        own = me * E_loc
        train = any(ctx.needs_input_grad)
        dev = x.device
        B = ep.buffers(T, C, k, E)
        u = ops.dwconv7(x, Fn._taps(dww), dwb)
        v = B['v'].view(T, C)
        _, stats = ops.layernorm_fwd(u, lnw, lnb, eps, tokens=T, C=C, out=v, save_stats=train)
        r, plan, slot_of, pair_token = Fn.route(v, wp, bp, sim, tau, w_noise, noise, T=T, C=C, E=E, k=k, save=train)
        R_s, cap = plan['max_rows'], B['cap']
        B['pair'][:R_s].copy_(pair_token)
        meta = torch.stack([plan['counts'], plan['seg_begin']]).contiguous()
        allm = torch.empty((Wn, 2, E), device=dev, dtype=torch.int32)
        dist.all_gather_into_tensor(allm, meta, group=ep.group)      # also orders "v / pair list written" before peer reads
        P = device_plan(ep, allm, plan['tile_group'], plan['num_m_tiles'], pair_token, E, R_s, cap)   # no host sync
        grouped = (P['tile_group'], P['num_tiles'])
        # every expert-side kernel runs over the fixed `cap` row space; the live tile count / segments come from the device
        xr = ops.gather_rows_peer(B['v_ptrs'], P['src_rank'], P['src_slot'], rows=cap, Cc=C, token_lists=B['pair_ptrs'])
        h, _ = Fn.expert_ffn_fwd(xr, w1s[own], b1s[own], w2s[own], b2s[own], packs, rows=cap, grouped=grouped,
                                 out=B['o'][:cap * C].view(cap, C))
        ep.barrier()                                                 # every rank's expert outputs are complete
        o = ops.gather_rows_peer(B['o_ptrs'], P['comb_rank'], P['comb_row'], rows=R_s, Cc=C)
        out, y = ops.moe_combine(o, slot_of, r['top_idx'], r['top_gate'], gamma, x.view(T, C), row_scale, T=T, Cc=C, k=k,
                                 want_y=record is not None)
        if record is not None:
            record.append(dict(v=v.clone(), top_idx=r['top_idx'], top_gate=r['top_gate'], importance=plan['importance'],
                               load=plan['load'], loss=plan['loss'], y=y, counts=plan['counts']))
        if train:
            # v lives in the symmetric buffer that the next layer of this shape overwrites: save a copy
            ctx.save_for_backward(*Fn.router_saved(r, plan, sim, tau, noise, w_noise), x, u, stats, v.clone(), h, xr, o, dww,
                                  lnw, gamma, wp, row_scale, slot_of, w1s[own], w2s[own])
            ctx.P, ctx.B, ctx.ep = P, B, ep
            ctx.E, ctx.k, ctx.R_s, ctx.own, ctx.E_loc = E, k, R_s, own, E_loc
            ctx.packs = packs
        return out.view(N, H, W_, C), plan['loss'].reshape(())

    @staticmethod
    def backward(ctx, dout, dloss):
        saved = ctx.saved_tensors
        router = saved[:Fn.ROUTER_SAVED]
        x, u, stats, v, h, xr, o, dww, lnw, gamma, wp, rs, slot_of, w1, w2 = saved[Fn.ROUTER_SAVED:]
        top_idx, top_gate = router[:2]
        P, B, ep = ctx.P, ctx.B, ctx.ep
        E, k, R_s, own, E_loc = ctx.E, ctx.k, ctx.R_s, ctx.own, ctx.E_loc
        N, H, W_, C = x.shape
        T = N * H * W_
        dev = x.device
        cap = P['cap']
        dout = dout.contiguous()
        dz = dout.view(T, C)
        grouped, segs = (P['tile_group'], P['num_tiles']), (P['seg_begin'], P['seg_end'])
        # combine backward on the source rank; d_o rows go to the symmetric buffer the expert ranks pull from (every live
        # slot is written, padding slots are never read: the expert side gathers through its source lists)
        d_o = B['do'][:R_s * C].view(R_s, C)
        dgamma = torch.zeros((C,), device=dev, dtype=torch.float32)
        dgate = ops.moe_combine_bwd(dz, o, slot_of, top_idx, top_gate, gamma, rs, d_o, dgamma, T=T, Cc=C, k=k)
        ep.barrier()                                                 # every rank's d_o rows are complete
        # gradients exist for the OWNED experts only (the others return None and stay out of the DDP buckets)
        dor = ops.gather_rows_peer(B['do_ptrs'], P['src_rank'], P['src_slot'], rows=cap, Cc=C)
        dxp, dw1s, db1s, dw2s, db2s = Fn.expert_ffn_bwd(dor, h, xr, w1, w2, ctx.packs, rows=cap, grouped=grouped, segs=segs,
                                                        groups=E_loc, dxp=B['dxp'][:cap * C].view(cap, C))
        ep.barrier()                                                 # every rank's d_x rows are complete
        dxp_l = ops.gather_rows_peer(B['dxp_ptrs'], P['comb_rank'], P['comb_row'], rows=R_s, Cc=C)
        dv_r, dwp, dbp, dsim, dtau, dwn = Fn.router_backward(router, v, wp, dgate, dloss, ctx.packs.get('wp_t'))
        dv = ops.gather_sum(dxp_l, slot_of, dv_r, T=T, Cc=C, k=k)
        dx, ddww, ddwb, dlnw, dlnb = Fn._block_front_bwd(dv, dout, x, u, stats, dww, lnw)
        if ep.average_grads:                  # what DDP's mean over ranks does to every other gradient
            for t in (dw1s, db1s, dw2s, db2s):
                t.mul_(1.0 / ep.world)

        def mine(t):
            return [t[e - own] if own <= e < own + E_loc else None for e in range(E)]
        grads_e = mine(dw1s) + mine(db1s) + mine(dw2s) + mine(db2s)
        return (dx, ddww, ddwb, dlnw, dlnb, dgamma, dwp, dbp, dsim, dtau, dwn, None, None, None, None, None, None, None, None,
                None, *grads_e)


def enable_expert_parallel(backbone, group=None, capacity_factor=2.0, average_grads=True):
    """Switch every MoE ConvNeXtBlock of ``backbone`` to the expert-parallel path.  Call on every rank of ``group`` after
    the process group exists; forward passes then allocate the symmetric buffers collectively.  Wrap the model in DDP with
    ``ddp_ignored_parameters(backbone)`` excluded (``DistributedDataParallel._set_params_and_buffers_to_ignore_for_model``):
    owned-expert gradients are already the DDP mean (average_grads), the others are None."""
    from .backbone import ConvNeXtBlock
    ctx = EPContext(group, capacity_factor, average_grads)
    n = 0
    for name, m in backbone.named_modules():
        if isinstance(m, ConvNeXtBlock) and m.MoE_cfg is not None:
            if m.ffn.num_experts % ctx.world:
                raise ValueError(f'{name}: num_experts={m.ffn.num_experts} is not divisible by world size {ctx.world}')
            m._ep = ctx
            m._ep_key = name
            n += 1
    backbone._ep_ctx = ctx
    return n


def ddp_ignored_parameters(backbone, prefix=''):
    """Names (as DDP sees them under ``prefix``) of every expert parameter: they never enter a gradient bucket."""
    return [prefix + n for n, _ in backbone.named_parameters() if '.ffn.experts.' in n]
