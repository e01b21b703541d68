"""Geographic partition of a world across the GPUs of one box (one process per GPU).

The reference has no multi-GPU code (SURVEY.md §2.1); this is the domain decomposition BASELINE.json's north
star asks for.  Agents are numbered area-contiguously, so rank r owns a contiguous agent range (cut where no
household-like group is split) and the groups its agents attend.  A step then runs in two stages
(``gj_step_params.stage``): every rank forms the partial sums of its groups from its own members, the sums of the
groups that straddle partitions ("boundary groups": commuter companies, schools, universities, leisure venues at
partition borders) are all-reduced over NCCL/NVLink in one packed buffer, and everything after that (gather,
exp, Gumbel-softmax draw, state update, symptoms) is rank-local.  The backward mirrors it with the cotangent
sums.  Each boundary group is *owned* by the lowest rank attending it, which alone adds its term to d/dbeta
(``gj_world_desc.dbeta_w``); summing the ranks' log-beta gradients gives the gradient of the whole world.
The Philox counter is the global agent id (``agent_offset``), so a partitioned run draws the same noise as the
unpartitioned one.
"""
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np
import torch

from .world import HeteroData, RANGE_MAX_GROUP, TIER_CELL, TIER_GENERIC, TIER_RANGE, ToUndirected


@dataclass
class Partition:
    rank: int
    world_size: int
    bounds: List[int]                      # world_size + 1 global agent cut points
    n_global_agents: int
    types: List[str]
    local_groups: Dict[str, torch.Tensor]  # type -> global ids of this rank's groups (ascending) = local id order
    n_boundary: Dict[str, int]             # type -> number of groups attended by >= 2 ranks (same on every rank)
    touch_pos: Dict[str, torch.Tensor]     # type -> positions of this rank's boundary groups in the global boundary list
    touch_lid: Dict[str, torch.Tensor]     # type -> their local group ids
    owned: Dict[str, torch.Tensor]         # type -> [G_local] bool: this rank is the lowest one attending the group
    process_group: object = None
    attend: Dict[str, torch.Tensor] = field(default_factory=dict)   # type -> [n_boundary] bit mask of the attending ranks

    @property
    def agent_lo(self):
        return self.bounds[self.rank]

    @property
    def agent_hi(self):
        return self.bounds[self.rank + 1]


def _slice_agents(v, lo, hi, n):
    if torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] == n:
        return v[lo:hi].clone()
    if isinstance(v, np.ndarray) and v.ndim >= 1 and v.shape[0] == n:
        return v[lo:hi].copy()
    if isinstance(v, dict):
        return {k: _slice_agents(x, lo, hi, n) for k, x in v.items()}
    return v


def partition_bounds(data: HeteroData, world_size: int) -> List[int]:
    """Equal-size agent ranges, each cut moved forward to the next agent at which no household-like group (every
    agent in at most one group, groups = short runs of consecutive agents) is split."""
    n = len(data["agent"].id)
    dev = data["agent"].age.device if torch.is_tensor(data["agent"].age) else "cpu"
    ok = torch.ones(n + 1, dtype=torch.bool, device=dev)
    for t in data.venue_types():
        ei = data["attends_" + t].edge_index
        if ei.shape[1] == 0:
            continue
        src, dst = ei[0], ei[1]
        if int(torch.bincount(src, minlength=n).max()) > 1:
            continue
        if int(torch.bincount(dst).max()) > RANGE_MAX_GROUP:
            continue
        gid = torch.full((n,), -1, dtype=torch.long, device=src.device)
        gid[src] = dst
        same = (gid[1:] == gid[:-1]) & (gid[1:] >= 0)      # agent a and a-1 share a group: no cut at a
        ok[1:n] &= ~same.to(ok.device)
    valid = torch.nonzero(ok).flatten()
    bounds = [0]
    for r in range(1, world_size):
        c = (n * r) // world_size
        j = int(torch.searchsorted(valid, torch.tensor([c], device=valid.device))[0])
        bounds.append(max(int(valid[min(j, valid.numel() - 1)]), bounds[-1]))
    bounds.append(n)
    return bounds


def partition_world(data: HeteroData, rank: int, world_size: int, bounds: Optional[List[int]] = None,
                    process_group=None) -> HeteroData:
    """This rank's part of ``data`` (a complete world, identical on every rank): its agents (every per-agent
    attribute sliced), the edges of its agents with group ids renumbered to the groups it attends, and the global
    ``people`` counts of those groups.  The partition record is attached as ``local._gj_partition``."""
    n = len(data["agent"].id)
    bounds = partition_bounds(data, world_size) if bounds is None else list(bounds)
    lo, hi = bounds[rank], bounds[rank + 1]
    types = data.venue_types()
    local = HeteroData()
    for key, v in data["agent"].items():
        local["agent"][key] = _slice_agents(v, lo, hi, n)
    cuts = None
    part = Partition(rank=rank, world_size=world_size, bounds=bounds, n_global_agents=n, types=types, local_groups={},
                     n_boundary={}, touch_pos={}, touch_lid={}, owned={}, process_group=process_group)
    for t in types:
        ei = data["attends_" + t].edge_index
        src, dst = ei[0], ei[1]
        dev = src.device
        G = len(data[t]["id"])
        if cuts is None or cuts.device != dev:
            cuts = torch.tensor(bounds[1:-1], dtype=torch.long, device=dev)
        # which ranks attend each group (from the complete edge list: the same answer on every rank)
        r_of = torch.bucketize(src, cuts, right=True)
        pairs = torch.unique(dst * world_size + r_of)
        pg, pr = pairs // world_size, pairs % world_size
        n_ranks = torch.bincount(pg, minlength=G)
        owner = torch.full((G,), world_size, dtype=torch.long, device=dev).scatter_reduce(0, pg, pr, reduce="amin")
        boundary_ids = torch.nonzero(n_ranks >= 2).flatten()                  # ascending global ids
        mine = pg[pr == rank]                                                 # ascending global ids of my groups
        sel = (src >= lo) & (src < hi)
        lsrc = src[sel] - lo
        ldst = torch.searchsorted(mine, dst[sel])
        local[t].id = torch.arange(mine.numel(), device=dev)
        people = torch.as_tensor(data[t]["people"])
        local[t].people = people.to(dev)[mine]
        for key, v in data[t].items():   # every other per-group attribute (a region label, ...) of my groups
            if key in ("id", "people"):
                continue
            if torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] == G:
                local[t][key] = v.to(dev)[mine]
            elif isinstance(v, np.ndarray) and v.ndim >= 1 and v.shape[0] == G:
                local[t][key] = v[mine.cpu().numpy()]
            else:
                local[t][key] = v
        local["agent", "attends_" + t, t].edge_index = torch.stack((lsrc, ldst))
        is_b = n_ranks[mine] >= 2
        lid = torch.nonzero(is_b).flatten()
        bits = torch.zeros(G, dtype=torch.long, device=dev).scatter_add_(0, pg, torch.ones_like(pr) << pr)
        part.attend[t] = bits[boundary_ids]
        part.local_groups[t] = mine
        part.n_boundary[t] = int(boundary_ids.numel())
        part.touch_lid[t] = lid
        part.touch_pos[t] = torch.searchsorted(boundary_ids, mine[lid])
        part.owned[t] = owner[mine] == rank
    if any(k[1].startswith("rev_") for k in data._edge_store_dict):
        local = ToUndirected()(local)
    local.__dict__["_gj_partition"] = part
    return local


def partition_from_blocks(block: HeteroData, process_group=None) -> HeteroData:
    """The rank's local world from ONE block of a world generated block-wise
    (``make_synthetic_world(..., block=(rank, world_size))``: local agent indices, global group ids) — the
    distributed counterpart of :func:`partition_world` for worlds no single GPU could hold.  Collectives (NCCL on
    GPUs, gloo on CPU): the block sizes (agent cut points), per group type the member counts of every rank's
    groups (``people`` = sum over ranks) and the attendance bitmaps (which ranks attend a group -> boundary list
    and owner).  The result is identical to ``partition_world(whole_world, rank, world_size, bounds)``."""
    import torch.distributed as dist

    rank, world_size, n_local = block.__dict__["_gj_block"]
    if dist.is_initialized():
        assert dist.get_world_size(process_group) == world_size and dist.get_rank(process_group) == rank
    elif world_size != 1:
        raise RuntimeError("partition_from_blocks needs an initialised process group")
    dev = block["agent"].age.device
    sizes = torch.zeros(world_size, dtype=torch.long, device=dev)
    sizes[rank] = n_local
    if world_size > 1:
        dist.all_reduce(sizes, group=process_group)
    bounds = [0] + [int(x) for x in torch.cumsum(sizes, 0).tolist()]
    types = block.venue_types()
    local = HeteroData()
    for key, v in block["agent"].items():
        local["agent"][key] = v
    part = Partition(rank=rank, world_size=world_size, bounds=bounds, n_global_agents=bounds[-1], types=types,
                     local_groups={}, n_boundary={}, touch_pos={}, touch_lid={}, owned={}, process_group=process_group)
    for t in types:
        ei = block["attends_" + t].edge_index
        src, gid = ei[0], ei[1]
        G = int(block[t].n_global)
        cnt = torch.bincount(gid, minlength=G)
        if block[t].scope == "local" or world_size == 1:
            mine = torch.nonzero(cnt > 0).flatten() if block[t].scope != "local" else torch.arange(G, device=dev)
            people = cnt[mine]
            n_ranks_mine = torch.ones(mine.numel(), dtype=torch.long, device=dev)
            owner_mine = torch.full((mine.numel(),), rank, dtype=torch.long, device=dev)
            boundary_ids = torch.zeros(0, dtype=torch.long, device=dev)
            attend_b = torch.zeros(0, dtype=torch.long, device=dev)
        else:
            mask = (cnt > 0).to(torch.uint8)
            masks = [torch.empty_like(mask) for _ in range(world_size)]
            dist.all_gather(masks, mask, group=process_group)
            masks = torch.stack(masks)                                   # [R, G]
            n_ranks = masks.sum(0, dtype=torch.long)
            owner = torch.argmax(masks, dim=0)                           # first (lowest) rank attending the group
            dist.all_reduce(cnt, group=process_group)                    # people = members over the whole world
            mine = torch.nonzero(mask).flatten()
            people = cnt[mine]
            n_ranks_mine, owner_mine = n_ranks[mine], owner[mine]
            boundary_ids = torch.nonzero(n_ranks >= 2).flatten()
            shifts = torch.arange(world_size, device=dev).reshape(-1, 1)
            attend_b = (masks[:, boundary_ids].long() << shifts).sum(0)
            del masks, n_ranks, owner
        local[t].id = torch.arange(mine.numel(), device=dev)
        local[t].people = people
        local["agent", "attends_" + t, t].edge_index = torch.stack((src, torch.searchsorted(mine, gid)))
        lid = torch.nonzero(n_ranks_mine >= 2).flatten()
        part.local_groups[t] = mine
        part.n_boundary[t] = int(boundary_ids.numel())
        part.touch_lid[t] = lid
        part.touch_pos[t] = torch.searchsorted(boundary_ids, mine[lid])
        part.owned[t] = owner_mine == rank
        part.attend[t] = attend_b
    local.__dict__["_gj_partition"] = part
    return local


class BoundaryExchange:
    """Packs the sums of this rank's boundary groups, all-reduces them, and writes the totals back."""

    def __init__(self, part: Partition, world):
        self.part = part
        self.world = world
        self._regions = {}
        self._packs = {}
        self._peer = None          # gj_peer* once connected; False = not available (the NCCL path runs)
        self.mode = "NCCL all-reduce of the packed buffer"
        dev = world.device
        w = torch.zeros(world.n_groups, dtype=torch.float32, device=dev)
        for ti, t in enumerate(world.types):
            w[world.type_group_off[ti]:world.type_group_off[ti + 1]] = part.owned[t].to(dev, torch.float32)
        world.dbeta_w = w
        if not hasattr(world, "handle"):
            world.__dict__.pop("_desc", None)   # the descriptor carries the pointer (a native world patches its own)

    def regions(self, lean: bool, gen_base: int, nets):
        """(index into the group-sum buffers, index into the packed buffer, packed length) for this step:
        ``nets`` = [(type index, s_off)] in network order."""
        key = (lean, gen_base, tuple(nets))
        hit = self._regions.get(key)
        if hit is not None:
            return hit
        world, part = self.world, self.part
        dev = world.device
        offsets = []                                  # (type index, offset of the type's groups in the buffers)
        if lean:
            for ti in range(len(world.types)):
                if world.type_tier[ti] == TIER_GENERIC:
                    offsets.append((ti, gen_base + world.type_group_off[ti]))
            offsets += [(ti, off) for ti, off in nets if world.type_tier[ti] == TIER_CELL]
        else:
            offsets += [(ti, off) for ti, off in nets if world.type_tier[ti] != TIER_RANGE]
        src, dst, base = [], [], 0
        for ti, off in offsets:
            t = world.types[ti]
            src.append(part.touch_lid[t].to(dev) + off)
            dst.append(part.touch_pos[t].to(dev) + base)
            base += part.n_boundary[t]
        cat = lambda xs: torch.cat(xs) if xs else torch.zeros(0, dtype=torch.long, device=dev)  # noqa: E731
        src, dst = cat(src), cat(dst)
        inv = torch.full((base,), -1, dtype=torch.int32, device=dev)   # pack position -> entry of the sum buffers
        inv[dst] = src.to(torch.int32)
        # which ranks attend each packed group (peer-memory exchange: where to store, whom to add, in rank order)
        attend = cat([part.attend[world.types[ti]].to(dev) for ti, _ in offsets]) if part.attend else None
        if attend is not None:
            attend = attend.to(torch.int32)
        self._check_layout(base, [ti for ti, _ in offsets])
        mine = torch.sort(dst)[0].to(torch.int32)        # the packed positions this rank attends, ascending
        hit = (src, dst, base, inv, attend, mine)
        self._regions[key] = hit
        return hit

    def _check_layout(self, n_pack, type_order):
        """Every rank must exchange the same packed layout (ADVICE r1: tiers chosen per rank once gave packs of
        different length).  Collective, once per new region: compare (length, type order) across ranks."""
        import torch.distributed as dist

        if self.part.world_size == 1 or not dist.is_initialized():
            return
        sig = torch.tensor([n_pack] + list(type_order) + [-1] * (8 - len(type_order)), dtype=torch.long)
        if dist.get_backend(self.part.process_group) == "nccl":
            sig = sig.to(self.world.device)
        both = torch.stack((sig, -sig))
        dist.all_reduce(both, op=dist.ReduceOp.MAX, group=self.part.process_group)
        if not torch.equal(both[0], -both[1]):
            raise RuntimeError(f"boundary exchange layout differs between ranks: this rank packs {sig.tolist()}")

    def _peer_context(self, device, n_needed=0):
        """Connect the NVLink peer-memory exchange (gj_peer_*) on first use; False if it cannot be had on every rank
        (then the NCCL path runs).  GJ_PEER=0 in the environment forces NCCL."""
        import ctypes as C
        import os

        import torch.distributed as dist

        from . import _lib
        L = _lib.lib()
        if self._peer is not None:
            if self._peer is False or n_needed <= self._peer_capacity:
                return self._peer
            # a packed layout larger than the buffers (e.g. one entry per NETWORK of a shared edge type): every rank
            # sees the same n_needed (regions() checks the layout across ranks), so all of them reconnect together
            torch.cuda.synchronize(device)
            dist.barrier(group=self.part.process_group)
            L.gj_peer_destroy(self._peer)
            self._peer = None
        part = self.part
        ok, peer = 1, C.c_void_p()
        why = ""
        capacity = max(int(sum(part.n_boundary.values())), int(n_needed))
        self._peer_capacity = capacity
        if os.environ.get("GJ_PEER", "1") == "0" or part.world_size > 32 or not part.attend:
            ok, why = 0, "disabled"
        handles = torch.zeros(part.world_size, 64, dtype=torch.uint8, device=device)
        with torch.cuda.device(device):
            if ok:
                if L.gj_peer_create(part.rank, part.world_size, capacity, C.byref(peer)) != 0:
                    ok, why = 0, L.gj_last_error().decode()
            if ok:
                buf = (C.c_uint8 * 64)()
                if L.gj_peer_handle(peer, buf) != 0:
                    ok, why = 0, L.gj_last_error().decode()
                else:
                    handles[part.rank] = torch.tensor(list(buf), dtype=torch.uint8).to(device)
            flag = torch.tensor([ok], device=device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=part.process_group)
            if int(flag) == 1:
                dist.all_reduce(handles, group=part.process_group)       # every row is zero except its owner's
                host = handles.cpu().contiguous()
                if L.gj_peer_connect(peer, C.c_void_p(host.data_ptr())) != 0:
                    ok, why = 0, L.gj_last_error().decode()
                flag = torch.tensor([ok], device=device)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=part.process_group)
            torch.cuda.synchronize(device)
            dist.barrier(group=part.process_group)
        if int(flag) == 1:
            self._peer = peer
            self.mode = "NVLink peer-memory stores + flags, one kernel (gj_peer_exchange)"
        else:
            self._peer = False
            self.mode = "NCCL all-reduce of the packed buffer" + (f" (peer memory unavailable: {why})" if why else "")
        return self._peer

    def check(self):
        """Raise if a peer did not arrive at an exchange in time (``gj_peer_status``; the kernel then carried on with
        incomplete sums rather than hang the GPU).  Synchronises the device: call it between windows, not per step."""
        if self._peer:
            from . import _lib
            with torch.cuda.device(self.world.device):
                torch.cuda.synchronize(self.world.device)
                if _lib.lib().gj_peer_status(self._peer) != 0:
                    raise _lib.GradJuneLibraryError("boundary exchange: " + _lib.lib().gj_last_error().decode())

    def exchange(self, buffers, region):
        """In place: every buffer's boundary entries become the sum over ranks.  On a GPU this is one pack
        kernel, one NCCL all-reduce of the packed [2, n_boundary] buffer and one unpack kernel."""
        import torch.distributed as dist

        src, dst, n, inv, attend, mine = region
        if n == 0 or self.part.world_size == 1:
            return
        a, b = buffers
        if a.is_cuda:
            import ctypes as C

            from . import _lib
            L = _lib.lib()
            peer = self._peer_context(a.device, n) if attend is not None else False
            if peer:
                st = C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream)
                with torch.cuda.device(a.device):
                    _lib.check(L.gj_peer_exchange(peer, n, inv.data_ptr(), attend.data_ptr(), a.data_ptr(), b.data_ptr(),
                                                  mine.numel(), mine.data_ptr(), st), "gj_peer_exchange")
                return
            pack = self._packs.get(n)
            if pack is None:
                pack = self._packs[n] = torch.empty(2, n, dtype=torch.float32, device=a.device)
            st = C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream)
            with torch.cuda.device(a.device):
                _lib.check(L.gj_boundary_pack(n, inv.data_ptr(), a.data_ptr(), b.data_ptr(), pack.data_ptr(), st),
                           "gj_boundary_pack")
                dist.all_reduce(pack, group=self.part.process_group)
                _lib.check(L.gj_boundary_unpack(n, inv.data_ptr(), pack.data_ptr(), a.data_ptr(), b.data_ptr(), st),
                           "gj_boundary_unpack")
            return
        pack = torch.zeros(len(buffers), n, dtype=torch.float32, device=a.device)   # host-logic tests (gloo)
        for i, buf in enumerate(buffers):
            pack[i, dst] = buf[src]
        dist.all_reduce(pack, group=self.part.process_group)
        for i, buf in enumerate(buffers):
            buf[src] = pack[i, dst]


class _AllReduceSum(torch.autograd.Function):
    """Sum over ranks of a tensor every rank then uses in the same loss: the cotangent passes through."""

    @staticmethod
    def forward(ctx, x, group):
        import torch.distributed as dist

        y = x.clone()
        dist.all_reduce(y, group=group)
        return y

    @staticmethod
    def backward(ctx, g):
        return g, None


def all_reduce_sum(x, part: Optional[Partition]):
    if part is None or part.world_size == 1:
        return x
    return _AllReduceSum.apply(x, part.process_group)


def label_union(values: np.ndarray, part: Optional[Partition]) -> np.ndarray:
    """Sorted union over the ranks of each rank's distinct label values (one all-gather): every rank of a partitioned
    world then has the same result columns."""
    if part is None or part.world_size == 1:
        return np.unique(values)
    import torch.distributed as dist

    gathered = [None] * part.world_size
    dist.all_gather_object(gathered, np.asarray(values), group=part.process_group)
    return np.unique(np.concatenate(gathered))


def exchange_for(data, world):
    """The BoundaryExchange of a partitioned world (cached on the data object), or None."""
    part = data.__dict__.get("_gj_partition")
    if part is None:
        return None
    cache = data.__dict__.setdefault("_gj_cache", {})
    hit = cache.get("exchange")
    if hit is None or hit.world is not world:
        hit = BoundaryExchange(part, world)
        cache["exchange"] = hit
    return hit
