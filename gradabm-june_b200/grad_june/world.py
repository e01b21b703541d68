"""World container and device layout.

``HeteroData`` is a torch_geometric-free stand-in that supports exactly the access patterns the
reference uses on its world object (runner.py:65-136, infection_networks/base.py:30-45):
``data["agent"].age``, ``data["agent"]["age"]``, ``data["agent","attends_school","school"].edge_index``,
``data["attends_school"]``, ``data["rev_attends_school"]``, ``data["school"]["people"]``,
``data["results"]``, ``del data["rev_attends_school"]`` and ``.to(device)``.  Reference pickles
(e.g. test/data/data.pkl) load into it through :func:`load_world`.

:func:`build_csr` turns the reference's unsorted int64 ``[2, E]`` edge lists into the CSR-sorted layout
the kernels read (``gj_world_desc`` in include/gradjune_b200.h); it is plain torch so that it runs on
the GPU for England-scale worlds and on the CPU for tests.
"""
import io
import pickle
import sys
from typing import Dict, List, Optional

import numpy as np
import torch

MAX_TYPES = 8


# --------------------------------------------------------------------------------------
# container
# --------------------------------------------------------------------------------------
class _Store:
    def __init__(self, key=None):
        object.__setattr__(self, "_mapping", {})
        object.__setattr__(self, "_key", key)

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        mapping = self.__dict__.get("_mapping", {})
        if name in mapping:
            return mapping[name]
        raise AttributeError(f"{type(self).__name__} {self.__dict__.get('_key')!r} has no attribute {name!r}")

    def __setattr__(self, name, value):
        self._mapping[name] = value

    def __getitem__(self, name):
        return self._mapping[name]

    def __setitem__(self, name, value):
        self._mapping[name] = value

    def __delitem__(self, name):
        del self._mapping[name]

    def __contains__(self, name):
        return name in self._mapping

    def keys(self):
        return self._mapping.keys()

    def items(self):
        return self._mapping.items()

    def __setstate__(self, state):  # torch_geometric storage pickles: {"_mapping", "_parent", "_key"}
        object.__setattr__(self, "_mapping", dict(state.get("_mapping", {})))
        object.__setattr__(self, "_key", state.get("_key"))

    def __getstate__(self):
        return {"_mapping": self._mapping, "_key": self._key}

    def __repr__(self):
        return f"{type(self).__name__}({self._key!r}: {list(self._mapping)})"


class NodeStorage(_Store):
    pass


class EdgeStorage(_Store):
    pass


class GlobalStorage(_Store):
    pass


def _move(v, device):
    if torch.is_tensor(v):
        return v.to(device)
    if isinstance(v, dict):
        return {k: _move(x, device) for k, x in v.items()}
    return v


class HeteroData:
    def __init__(self):
        self.__dict__["_global_store"] = GlobalStorage("global")
        self.__dict__["_node_store_dict"] = {}
        self.__dict__["_edge_store_dict"] = {}
        self.__dict__["_gj_cache"] = {}

    def __setstate__(self, state):
        self.__dict__.update(state)
        self.__dict__.setdefault("_gj_cache", {})

    def __getstate__(self):
        return {k: v for k, v in self.__dict__.items() if k != "_gj_cache"}

    def _edge_key(self, rel):
        for k in self._edge_store_dict:
            if k[1] == rel:
                return k
        return None

    def __getitem__(self, key):
        if isinstance(key, tuple):
            if key not in self._edge_store_dict:
                self._edge_store_dict[key] = EdgeStorage(key)
            return self._edge_store_dict[key]
        ek = self._edge_key(key)
        if ek is not None:
            return self._edge_store_dict[ek]
        if key in self._global_store:
            return self._global_store[key]
        if key not in self._node_store_dict:
            self._node_store_dict[key] = NodeStorage(key)
        return self._node_store_dict[key]

    def __setitem__(self, key, value):
        self._global_store[key] = value

    def __delitem__(self, key):
        if isinstance(key, tuple):
            del self._edge_store_dict[key]
            return
        ek = self._edge_key(key)
        if ek is not None:
            del self._edge_store_dict[ek]
        elif key in self._node_store_dict:
            del self._node_store_dict[key]
        else:
            del self._global_store[key]

    def __contains__(self, key):
        return (self._edge_key(key) is not None or key in self._node_store_dict or key in self._global_store)

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        gs = self.__dict__.get("_global_store")
        if gs is not None and name in gs:
            return gs[name]
        raise AttributeError(name)

    @property
    def node_types(self):
        return list(self._node_store_dict)

    @property
    def edge_types(self):
        return list(self._edge_store_dict)

    def to(self, device):
        for store in [*self._node_store_dict.values(), *self._edge_store_dict.values(), self._global_store]:
            for k, v in list(store.items()):
                store[k] = _move(v, device)
        self._gj_cache.clear()
        return self

    def venue_types(self) -> List[str]:
        """Edge types present, in insertion order: 'school' for ('agent','attends_school','school')."""
        return [k[1][len("attends_"):] for k in self._edge_store_dict if k[1].startswith("attends_")]


class ToUndirected:
    """Adds (dst, "rev_"+rel, src) edge stores holding ``edge_index.flip(0)`` (same edge order)."""

    def __call__(self, data):
        for (src, rel, dst) in list(data._edge_store_dict):
            if rel.startswith("rev_"):
                continue
            data[(dst, "rev_" + rel, src)].edge_index = data._edge_store_dict[(src, rel, dst)].edge_index.flip(0)
        return data


class _WorldUnpickler(pickle.Unpickler):
    """Reads reference pickles without torch_geometric: its classes map onto the stand-ins above."""

    _MAP = {"HeteroData": HeteroData, "NodeStorage": NodeStorage, "EdgeStorage": EdgeStorage,
            "GlobalStorage": GlobalStorage, "BaseStorage": GlobalStorage}

    def find_class(self, module, name):
        if module.startswith("torch_geometric"):
            if name in self._MAP:
                return self._MAP[name]
            raise pickle.UnpicklingError(f"unsupported torch_geometric class {module}.{name}")
        return super().find_class(module, name)


def load_world(path_or_file):
    """Load a world pickle written either by the reference (torch_geometric HeteroData) or by us."""
    if hasattr(path_or_file, "read"):
        return _WorldUnpickler(path_or_file).load()
    with open(path_or_file, "rb") as f:
        return _WorldUnpickler(f).load()


def world_from_arrays(arrays: Dict[str, np.ndarray], types: List[str], device="cpu") -> HeteroData:
    """Build a world from the plain-array form used by tests/golden/sample_world.npz."""
    data = HeteroData()
    n = len(arrays["age"])
    data["agent"].id = torch.arange(n)
    data["agent"].age = torch.as_tensor(np.asarray(arrays["age"]).astype(np.int64))
    data["agent"].sex = torch.as_tensor(np.asarray(arrays["sex"]).astype(np.int64))
    if "ethnicity" in arrays:
        data["agent"].ethnicity = np.asarray(arrays["ethnicity"])
    for t in types:
        ng = int(arrays[f"{t}_ngroups"])
        data[t].id = torch.arange(ng)
        data[t].people = torch.as_tensor(np.asarray(arrays[f"{t}_people"]).astype(np.int64))
        ei = np.stack([arrays[f"{t}_src"], arrays[f"{t}_dst"]]).astype(np.int64)
        data["agent", "attends_" + t, t].edge_index = torch.as_tensor(ei)
    data = ToUndirected()(data)
    return data.to(device)


def group_labels(data: HeteroData, edge_type: str, by: str) -> np.ndarray:
    """The region of every group of ``edge_type`` (numpy array, one entry per group in id order): the group attribute
    ``data[edge_type][by]`` when the world carries it, else derived from the members: the value of
    ``data["agent"][by]`` that most of the group's members carry, ties going to the smallest value (a group without
    members takes the smallest value of the world).  The derivation needs every member of a group, so it runs on a
    complete world: a partitioned world whose groups carry no ``by`` raises."""
    store = data[edge_type]
    G = len(store["id"])
    if by in store:
        v = store[by]
        a = v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)
        if a.ndim != 1 or a.shape[0] != G:
            raise ValueError(f"data[{edge_type!r}].{by} must hold one value per group ({G}), got shape {a.shape}")
        return a
    if "_gj_partition" in data.__dict__ or "_gj_block" in data.__dict__:
        raise ValueError(f"the groups of {edge_type!r} carry no {by!r}: a rank of a partitioned world cannot see all of a "
                         f"group's members; set data[{edge_type!r}].{by} on the complete world before partitioning")
    v = data["agent"][by]
    agent = v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)
    ei = data["attends_" + edge_type].edge_index.detach().cpu().numpy()
    n = len(data["agent"].id)
    if agent.ndim != 1 or agent.shape[0] not in (1, n):
        raise ValueError(f"data['agent'].{by} must hold one value per agent ({n}), got shape {agent.shape}")
    values, codes = np.unique(np.broadcast_to(agent, (n,)), return_inverse=True)
    L = len(values)
    pair, count = np.unique(ei[1].astype(np.int64) * L + codes[ei[0]], return_counts=True)
    grp, code = pair // L, pair % L
    # per group: the largest count, then the smallest code (lexsort: last key first)
    idx = np.lexsort((code, -count, grp))
    first = np.ones(idx.shape[0], dtype=bool)
    first[1:] = grp[idx][1:] != grp[idx][:-1]
    out = np.zeros(G, dtype=np.int64)
    out[grp[idx][first]] = code[idx][first]
    return values[out]


# --------------------------------------------------------------------------------------
# CSR layout
# --------------------------------------------------------------------------------------
TIER_GENERIC, TIER_RANGE, TIER_CELL = 0, 1, 2
TILE_AGENTS = 1024          # agents per CTA tile of the agent-major kernels (== GJ_TILE_AGENTS)
RANGE_MAX_GROUP = 64        # range tier: every agent re-sums its (small) group from its neighbours
CELL_MIN_MEAN_AGENTS = 64   # cell tier only pays when cells are much larger than a warp
CELL_MAX_GROUPS = 16
SCATTER_MAX_GROUP = 32768   # == GJ_SCATTER_MAX_GROUP: larger generic groups are "giant" (summed group-major in the forward)


class DeviceWorld:
    """Device arrays of the world + the ctypes descriptor handed to the library.

    Every edge type is stored in the cheapest of three layouts (``type_tier``):
      * RANGE  — each group is a contiguous, ascending run of agent ids and every agent belongs to at most
        one group (households after area-contiguous numbering): per agent one packed (offset, size) word and
        the group's contact probability; group sums are re-formed in-stream from neighbouring agents, there
        is no group-major pass and no per-group buffer;
      * CELL   — consecutive agents share the same ordered list of groups (leisure: everybody of a super-area
        attends the same k nearest venues): agents -> tile partial sums -> cells -> groups, so the per-edge
        work of the 3 leisure edges per agent collapses to one streaming pass;
      * GENERIC — CSR in both orientations (companies, schools, ...; any world that is not laid out as above).
    """

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def desc(self):
        from . import _lib

        d = self.__dict__.get("_desc")
        if d is not None:
            return d
        d = _lib.WorldDesc()
        d.n_agents, d.n_groups, d.n_edges, d.n_types = self.n_agents, self.n_groups, self.n_edges, len(self.types)
        for i, off in enumerate(self.type_group_off):
            d.type_group_off[i] = off
        for name in ("am_ptr", "am_ent", "gm_ptr", "gm_agent", "pc", "cls", "small_groups", "chunk_group",
                     "chunk_begin", "chunk_end", "chunk_part", "big_groups", "big_part_ptr", "tile_begin", "tile_flags",
                     "ent1"):
            setattr(d, name, getattr(self, name).data_ptr())
        d.n_small, d.n_chunks = self.small_groups.numel(), self.chunk_group.numel()
        d.n_big, d.n_parts = self.big_groups.numel(), self.n_parts
        d.n_giant_chunks, d.n_giant_big = self.__dict__.get("n_giant_chunks", 0), self.__dict__.get("n_giant_big", 0)
        d.n_tiles = self.tile_begin.numel() - 1
        cell_off = 0
        for ti in range(len(self.types)):
            d.type_tier[ti] = self.type_tier[ti]
            d.cell_off[ti] = cell_off
            if self.type_tier[ti] == TIER_RANGE:
                d.range_slot[ti] = self.range_slot[ti].data_ptr()
                d.range_pc[ti] = self.range_pc[ti].data_ptr()
                d.range_pc_from_size[ti] = 1 if self.__dict__.get("range_pc_from_size", {}).get(ti) else 0
            elif self.type_tier[ti] == TIER_CELL:
                c = self.cells[ti]
                d.n_cells[ti] = c["n_cells"]
                for name in ("tile_cell", "cell_tile_ptr", "cell_grp_ptr", "cell_grp", "grp_cell_ptr", "grp_cell"):
                    getattr(d, name)[ti] = c[name].data_ptr()
                cell_off += c["n_cells"]
        d.n_cells_total = cell_off
        if self.__dict__.get("dbeta_w") is not None:
            d.dbeta_w = self.dbeta_w.data_ptr()
        if self.__dict__.get("orig_id") is not None:
            d.orig_id = self.orig_id.data_ptr()
        self.__dict__["_desc"] = d
        return d


def p_contact(people: torch.Tensor) -> torch.Tensor:
    """clamp(1 / (people - 1), 0, 1) evaluated like infection_networks/base.py:64-69 (fp32)."""
    one = torch.tensor(1.0, device=people.device)
    zero = torch.tensor(0.0, device=people.device)
    return torch.maximum(torch.minimum(1.0 / (people - 1), one), zero).to(torch.float32)


def _u32(t):
    """uint32 values stored as int32 bit patterns (torch has no general uint32 support)."""
    t = t.to(torch.int64)
    return (((t + (1 << 31)) % (1 << 32)) - (1 << 31)).to(torch.int32).contiguous()


def _padded(t, slack=32):
    """Same tensor with `slack` readable elements behind it: the kernels fetch tiles with 16-byte-granular bulk
    copies that may run a few elements past the logical end."""
    buf = torch.zeros(t.numel() + slack, dtype=t.dtype, device=t.device)
    buf[: t.numel()] = t
    return buf[: t.numel()]


def _ptr_from_counts(counts):
    ptr = torch.zeros(counts.numel() + 1, dtype=torch.long, device=counts.device)
    ptr[1:] = torch.cumsum(counts, 0)
    return ptr


def _try_range_tier(n_agents, src, dst, n_groups, pc_t):
    """RANGE layout if every agent has <= 1 edge and every group is a contiguous ascending id run."""
    E = src.numel()
    dev = src.device
    deg = torch.bincount(src, minlength=n_agents)
    if E == 0 or int(deg.max()) > 1:
        return None
    size = torch.bincount(dst, minlength=n_groups)
    if int(size.max()) > RANGE_MAX_GROUP:
        return None
    _, perm = torch.sort(dst, stable=True)
    members = src[perm]
    ptr = _ptr_from_counts(size)
    gid = dst[perm]
    first = members[ptr[:-1].clamp(max=E - 1)]          # first member of each group (garbage for empty groups)
    offset = members - first[gid]
    if not bool((offset == torch.arange(E, device=dev) - ptr[gid]).all()):
        return None
    slot = torch.full((n_agents,), 0xFFFFFFFF, dtype=torch.long, device=dev)
    slot[members] = (offset << 16) | size[gid]
    rpc = torch.zeros(n_agents, dtype=torch.float32, device=dev)
    rpc[members] = pc_t[gid]
    from_size = bool(torch.equal(pc_t[gid], p_contact(size[gid])))     # `people` is the member count
    return {"range_slot": _padded(_u32(slot)), "range_pc": _padded(rpc.contiguous()), "pc_from_size": from_size}


def _try_cell_tier(n_agents, src, dst, n_groups):
    """CELL layout if long runs of consecutive agents share the same ordered group list."""
    E = src.numel()
    dev = src.device
    if E == 0:
        return None
    deg = torch.bincount(src, minlength=n_agents)
    if int(deg.max()) > CELL_MAX_GROUPS:
        return None
    _, perm = torch.sort(src, stable=True)
    s_sorted, d_sorted = src[perm], dst[perm]
    aptr = _ptr_from_counts(deg)
    pos = torch.arange(E, device=dev) - aptr[s_sorted]
    # exact comparison of each agent's ordered list with its predecessor's
    same_deg = torch.ones(n_agents, dtype=torch.bool, device=dev)
    same_deg[1:] = deg[1:] == deg[:-1]
    same_deg[0] = False
    prev_idx = (aptr[(s_sorted - 1).clamp(min=0)] + pos).clamp(max=E - 1)
    differs = (d_sorted != d_sorted[prev_idx]) & same_deg[s_sorted]
    n_diff = torch.zeros(n_agents, dtype=torch.long, device=dev).index_add_(0, s_sorted, differs.long())
    boundary = ~same_deg | (n_diff > 0)
    n_cells = int(boundary.sum())
    if n_cells * CELL_MIN_MEAN_AGENTS > n_agents:
        return None
    cell_start = torch.nonzero(boundary).flatten()
    cell_of_agent = torch.cumsum(boundary.long(), 0) - 1
    cdeg = deg[cell_start]
    cell_grp_ptr = _ptr_from_counts(cdeg)
    idx = torch.repeat_interleave(aptr[cell_start], cdeg) + (torch.arange(int(cdeg.sum()), device=dev)
                                                             - torch.repeat_interleave(cell_grp_ptr[:-1], cdeg))
    cell_grp = d_sorted[idx]
    cell_ids = torch.repeat_interleave(torch.arange(n_cells, device=dev), cdeg)
    _, gperm = torch.sort(cell_grp, stable=True)
    grp_cell = cell_ids[gperm]
    grp_cell_ptr = _ptr_from_counts(torch.bincount(cell_grp, minlength=n_groups))
    return {"n_cells": n_cells, "cell_start": cell_start, "cell_of_agent": cell_of_agent,
            "cell_grp_ptr": _u32(cell_grp_ptr), "cell_grp": _u32(cell_grp), "grp_cell_ptr": _u32(grp_cell_ptr),
            "grp_cell": _u32(grp_cell)}


def _degree_and_size(n_agents, ei, n_groups):
    E = ei.shape[1]
    if E == 0:
        return 0, 0
    return int(torch.bincount(ei[0], minlength=n_agents).max()), int(torch.bincount(ei[1], minlength=n_groups).max())


def tier_candidates(n_agents: int, types: List[str], edges: Dict[str, torch.Tensor], n_groups: Dict[str, int]):
    """Which edge type may use the RANGE tier and which the CELL tier (-> (range_type, cell_type), either may be None).

    The throughput-mode kernels take at most one range-tier network (the household re-sum over neighbouring agents)
    and run the cell tier for the leisure kinds only, and the reference itself addresses these two edge sets by
    name (``HouseholdNetwork`` -> "attends_household", every ``LeisureNetwork`` -> "attends_leisure",
    leisure_network.py:44-48,58-59).  So: RANGE = "household" if every agent has at most one such edge and no group
    exceeds ``RANGE_MAX_GROUP`` members, else the largest other type of that shape; CELL = "leisure" if no agent
    has more than ``CELL_MAX_GROUPS`` such edges.  Whether the tier is actually used is decided from the agent
    numbering by :func:`build_csr`; :func:`layout_order` computes the numbering that makes it so."""
    shape = {t: _degree_and_size(n_agents, edges[t], int(n_groups[t])) for t in types}
    cell_type = "leisure" if ("leisure" in types and 0 < shape["leisure"][0] <= CELL_MAX_GROUPS) else None
    ok = [t for t in types if t != cell_type and shape[t][0] == 1 and shape[t][1] <= RANGE_MAX_GROUP]
    range_type = None
    if "household" in ok:
        range_type = "household"
    elif ok:
        range_type = max(ok, key=lambda t: edges[t].shape[1])
    return range_type, cell_type


def _list_rank(n_agents, ei, n_groups):
    """Dense lexicographic rank of every agent's ORDERED group list (edge order; agents without an edge rank 0) and
    the number of distinct lists."""
    dev = ei.device
    src, dst = ei[0], ei[1]
    deg = torch.bincount(src, minlength=n_agents)
    _, perm = torch.sort(src, stable=True)
    s_sorted, d_sorted = src[perm], dst[perm]
    pos = torch.arange(src.numel(), device=dev) - _ptr_from_counts(deg)[s_sorted]
    rank = torch.zeros(n_agents, dtype=torch.long, device=dev)
    n_lists = 1
    for j in range(int(deg.max()) if src.numel() else 0):
        gj = torch.zeros(n_agents, dtype=torch.long, device=dev)
        sel = pos == j
        gj[s_sorted[sel]] = d_sorted[sel] + 1
        uniq, rank = torch.unique(rank * (int(n_groups) + 1) + gj, return_inverse=True)
        n_lists = int(uniq.numel())
    return rank, n_lists


def layout_order(n_agents: int, types: List[str], edges: Dict[str, torch.Tensor], n_groups: Dict[str, int]):
    """Agent renumbering that lets the world use the streaming layout tiers whatever order it was loaded in
    (SURVEY.md 7 "Random 4-byte gathers"; the reference's loaders number agents by area and age,
    june_world_loader/network_loader.py:30-44, so the members of a household are scattered over their area).

    Returns ``perm`` with ``perm[new] = old`` or None when the given numbering already has the layout.  Order:
    (1) the leisure cell — agents with the same ordered list of leisure groups, i.e. the same super-area — in
    lexicographic order of the lists, so that geography stays contiguous; (2) the household, placed in the cell of
    its first member; (3) the position of the agent's household edge in the edge list (members keep the reference's
    edge order, which the reference-order kernels sum in).  Agents without a household are singletons."""
    range_type, cell_type = tier_candidates(n_agents, types, edges, n_groups)
    if n_agents == 0 or (range_type is None and cell_type is None):
        return None
    dev = edges[types[0]].device
    ids = torch.arange(n_agents, device=dev)
    cell = torch.zeros(n_agents, dtype=torch.long, device=dev)
    n_cells = 1
    if cell_type is not None:
        cell, n_cells = _list_rank(n_agents, edges[cell_type], n_groups[cell_type])
    if range_type is not None:
        ei = edges[range_type]
        Gh = int(n_groups[range_type])
        hkey = Gh + ids                                     # singletons: one pseudo-household per agent
        hkey[ei[0]] = ei[1]
        epos = ei.shape[1] + ids
        epos[ei[0]] = torch.arange(ei.shape[1], device=dev)
    else:
        Gh, hkey, epos = 0, ids.clone(), ids
    n_keys = Gh + n_agents
    first = torch.full((n_keys,), int(epos.max()) + 1, dtype=torch.long, device=dev).scatter_reduce(
        0, hkey, epos, reduce="amin")
    hcell = torch.full((n_keys,), n_cells, dtype=torch.long, device=dev)
    is_first = epos == first[hkey]
    hcell[hkey[is_first]] = cell[is_first]                 # the cell of the household's first member
    base = torch.argsort(epos)                             # (3): members in edge order
    _, order = torch.sort((hcell[hkey] * n_keys + hkey)[base], stable=True)
    perm = base[order]
    if bool((perm == ids).all()):
        return None
    return perm


def _permute_agents(v, perm, n):
    if torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] == n:
        return v[perm.to(v.device)]
    if isinstance(v, np.ndarray) and v.ndim >= 1 and v.shape[0] == n:
        return v[perm.cpu().numpy()]
    if isinstance(v, dict):
        return {k: _permute_agents(x, perm, n) for k, x in v.items()}
    return v


def renumber_world(data: "HeteroData", perm: Optional[torch.Tensor] = None) -> "HeteroData":
    """The same world with its agents renumbered by :func:`layout_order` (or the given ``perm[new] = old``): every
    per-agent attribute is permuted, agent indices in the edge lists are rewritten (edge order unchanged), groups
    keep their ids.  ``data["agent"].original_index[new] = old`` records where each agent came from — the noise
    stream is keyed by it, so trajectories do not depend on the numbering — and :func:`original_order` maps
    per-agent results back.  Returns ``data`` itself when the numbering already has the layout."""
    n = len(data["agent"].id)
    types = data.venue_types()
    if perm is None:
        perm = layout_order(n, types, {t: data["attends_" + t].edge_index for t in types},
                            {t: len(data[t]["id"]) for t in types})
        if perm is None:
            return data
    perm = perm.long()
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(n, device=perm.device)
    prev = data["agent"]["original_index"] if "original_index" in data["agent"] else None
    for key, v in list(data["agent"].items()):
        data["agent"][key] = _permute_agents(v, perm, n)
    if prev is None:
        data["agent"].original_index = perm.clone()
    for (src, rel, dst), store in data._edge_store_dict.items():
        ei = store.edge_index
        row = 0 if src == "agent" else (1 if dst == "agent" else None)
        if row is None or ei.numel() == 0:
            continue
        ei = ei.clone()
        ei[row] = inv.to(ei.device)[ei[row]]
        store.edge_index = ei
    data._gj_cache.clear()
    return data


def layout_order_of(data: "HeteroData", values):
    """Per-agent ``values`` given in the order the world was loaded in -> the (renumbered) order of ``data``."""
    agent = data["agent"]
    if "original_index" not in agent:
        return values
    return _permute_agents(values, agent["original_index"], agent["original_index"].numel())


def original_order(data: "HeteroData", values: torch.Tensor) -> torch.Tensor:
    """Per-agent ``values`` of a renumbered world in the order the world was loaded in (differentiable)."""
    agent = data["agent"]
    if "original_index" not in agent or "_gj_partition" in data.__dict__:
        return values       # one part of a partitioned world keeps its local order: the caller assembles the parts
    cache = data.__dict__.setdefault("_gj_cache", {})
    oi = agent["original_index"]
    hit = cache.get("inverse_index")
    if hit is None or hit[0] is not oi:
        inv = torch.empty_like(oi)
        inv[oi] = torch.arange(oi.numel(), device=oi.device)
        cache["inverse_index"] = hit = (oi, inv)
    return values[hit[1].to(values.device)]


def build_csr(n_agents: int, types: List[str], edges: Dict[str, torch.Tensor], people: Dict[str, torch.Tensor],
              n_groups: Dict[str, int], age: torch.Tensor, sex: torch.Tensor, small_group: int, chunk: int,
              device, tiers: bool = True, orig_id: Optional[torch.Tensor] = None,
              want_tiers: Optional[Dict[str, int]] = None, scatter_max: int = SCATTER_MAX_GROUP) -> DeviceWorld:
    """``orig_id``: [n_agents] id of every agent in the numbering the world was loaded in (None = this one): the
    counter of the kernels' Philox stream.  ``want_tiers``: the tier to try per type (default: the policy of
    :func:`tier_candidates`; a partitioned world passes the tiers its ranks agreed on); a type whose structure
    does not fit the wanted tier is stored GENERIC."""
    if len(types) > MAX_TYPES:
        raise ValueError(f"at most {MAX_TYPES} edge types are supported")
    dev = torch.device(device)
    edges = {t: edges[t].to(dev) for t in types}
    if want_tiers is None:
        want_tiers = {}
        if tiers and n_agents > 0:
            range_type, cell_type = tier_candidates(n_agents, types, edges, n_groups)
            if range_type is not None:
                want_tiers[range_type] = TIER_RANGE
            if cell_type is not None:
                want_tiers[cell_type] = TIER_CELL
    offs = [0]
    for t in types:
        offs.append(offs[-1] + int(n_groups[t]))
    G = offs[-1]
    pc = torch.cat([p_contact(torch.as_tensor(people[t]).to(dev)) for t in types]) if types else torch.zeros(0, device=dev)
    if pc.numel() != G:
        raise ValueError("people arrays do not match the number of groups")
    type_tier, range_slot, range_pc, cells, range_from_size = [], {}, {}, {}, {}
    srcs, gkeys, ents = [], [], []
    n_edges_total = 0
    for ti, t in enumerate(types):
        ei = edges[t].to(dev)
        if ei.numel():
            if int(ei[0].max()) >= n_agents or int(ei[0].min()) < 0:
                raise ValueError(f"edge type {t}: agent index out of range")
            if int(ei[1].max()) >= n_groups[t] or int(ei[1].min()) < 0:
                raise ValueError(f"edge type {t}: group index out of range")
        if n_groups[t] >= (1 << 28):
            raise ValueError(f"edge type {t}: too many groups")
        n_edges_total += ei.shape[1]
        tier = TIER_GENERIC
        want = want_tiers.get(t, TIER_GENERIC) if (tiers and n_agents > 0) else TIER_GENERIC
        if want == TIER_RANGE:
            r = _try_range_tier(n_agents, ei[0], ei[1], int(n_groups[t]), pc[offs[ti]:offs[ti + 1]])
            if r is not None:
                tier, range_slot[ti], range_pc[ti] = TIER_RANGE, r["range_slot"], r["range_pc"]
                range_from_size[ti] = r["pc_from_size"]
        elif want == TIER_CELL:
            c = _try_cell_tier(n_agents, ei[0], ei[1], int(n_groups[t]))
            if c is not None:
                tier, cells[ti] = TIER_CELL, c
        type_tier.append(tier)
        if tier == TIER_GENERIC:
            srcs.append(ei[0])
            gkeys.append(ei[1] + offs[ti])
            ents.append(ei[1] + (ti << 28))
    if srcs:
        src, gkey, ent = torch.cat(srcs), torch.cat(gkeys), torch.cat(ents)
    else:
        src = gkey = ent = torch.zeros(0, dtype=torch.long, device=dev)
    E = src.numel()
    if n_edges_total >= (1 << 32) or n_agents >= (1 << 32):
        raise ValueError("world too large for 32-bit CSR offsets")
    # group-major: stable sort by global group id keeps the reference's edge order inside each group
    _, perm = torch.sort(gkey, stable=True)
    gm_agent = src[perm].to(torch.int32)
    size = torch.bincount(gkey, minlength=G) if E else torch.zeros(G, dtype=torch.long, device=dev)
    gm_ptr = _ptr_from_counts(size)
    del perm
    # agent-major: types were concatenated in order, so a stable sort by agent gives (type, edge order)
    _, perm = torch.sort(src, stable=True)
    am_ent = ent[perm].to(torch.int64)
    deg = torch.bincount(src, minlength=n_agents) if E else torch.zeros(n_agents, dtype=torch.long, device=dev)
    am_ptr = _ptr_from_counts(deg)
    del perm
    # one-entry-per-agent view for the throughput-mode kernels: global group id | none | "several: use the CSR"
    if G >= (1 << 31):
        raise ValueError("too many groups for the one-entry-per-agent view")
    if scatter_max < chunk:
        raise ValueError("scatter_max must be at least one chunk")
    ent1 = torch.full((n_agents,), 0xFFFFFFFF, dtype=torch.long, device=dev)
    if E:
        ent1[src] = gkey + ((size[gkey] > scatter_max).long() << 31)      # bit 31: a giant group
        ent1[deg > 1] = 0xFFFFFFFE
    age = age.to(dev).long()
    sex = sex.to(dev).long()
    if age.numel() and (int(age.min()) < 0 or int(age.max()) > 99 or int(sex.min()) < 0 or int(sex.max()) > 1):
        raise ValueError("age must be in [0, 99] and sex in {0, 1}")
    cls = (sex * 100 + age).to(torch.uint8)

    # work lists of the group-major passes (GENERIC types only: the other tiers have no group-major pass)
    generic_group = torch.zeros(G, dtype=torch.bool, device=dev)
    for ti in range(len(types)):
        if type_tier[ti] == TIER_GENERIC:
            generic_group[offs[ti]:offs[ti + 1]] = True
    gids = torch.arange(G, device=dev)
    small = gids[(size <= small_group) & generic_group]
    big_mask = (size > small_group) & generic_group
    giant = size > scatter_max
    bg = torch.cat((gids[big_mask & giant], gids[big_mask & ~giant]))     # giant groups lead the chunk lists
    n_giant_big = int((big_mask & giant).sum())
    nchunk = (size[bg] + chunk - 1) // chunk
    n_giant_chunks = int(nchunk[:n_giant_big].sum())
    chunk_group = torch.repeat_interleave(bg, nchunk)
    first = _ptr_from_counts(nchunk)
    within = torch.arange(chunk_group.numel(), device=dev) - torch.repeat_interleave(first[:-1], nchunk)
    chunk_begin = gm_ptr[chunk_group] + within * chunk
    chunk_end = torch.minimum(chunk_begin + chunk, gm_ptr[chunk_group + 1])
    multi = torch.repeat_interleave(nchunk > 1, nchunk)
    chunk_part = torch.full((chunk_group.numel(),), -1, dtype=torch.long, device=dev)
    n_parts = int(multi.sum())
    chunk_part[multi] = torch.arange(n_parts, device=dev)
    big_groups = bg[nchunk > 1]
    big_part_ptr = _ptr_from_counts(nchunk[nchunk > 1])

    # CTA tiles of the agent-major kernels: <= TILE_AGENTS consecutive agents inside one cell of every CELL type
    cuts = [torch.zeros(1, dtype=torch.long, device=dev)]
    for c in cells.values():
        cuts.append(c["cell_start"])
    seg_start = torch.unique(torch.cat(cuts)) if n_agents > 0 else torch.zeros(0, dtype=torch.long, device=dev)
    seg_end = torch.cat((seg_start[1:], torch.tensor([n_agents], device=dev))) if n_agents > 0 else seg_start
    ntile = (seg_end - seg_start + TILE_AGENTS - 1) // TILE_AGENTS
    tfirst = _ptr_from_counts(ntile)
    tw = torch.arange(int(ntile.sum()), device=dev) - torch.repeat_interleave(tfirst[:-1], ntile)
    tile_begin = torch.cat((torch.repeat_interleave(seg_start, ntile) + tw * TILE_AGENTS,
                            torch.tensor([n_agents], device=dev)))
    tile_flags = torch.zeros(tile_begin.numel() - 1, dtype=torch.long, device=dev)
    if tile_flags.numel():
        tile_flags[0] = 1
    for ti, c in cells.items():
        tc = c["cell_of_agent"][tile_begin[:-1]]
        tile_flags[1:] |= (tc[1:] != tc[:-1]).long()
    for ti, c in cells.items():
        c["tile_cell"] = _u32(c["cell_of_agent"][tile_begin[:-1]])
        c["cell_tile_ptr"] = _u32(torch.cat((torch.searchsorted(tile_begin[:-1].contiguous(), c["cell_start"]),
                                             torch.tensor([tile_begin.numel() - 1], device=dev))))
        del c["cell_of_agent"]

    return DeviceWorld(
        n_agents=n_agents, n_groups=G, n_edges=n_edges_total, n_generic_edges=E, types=list(types),
        type_group_off=offs, type_tier=type_tier, range_slot=range_slot, range_pc=range_pc, cells=cells,
        range_pc_from_size=range_from_size,
        group_size=size, am_ptr=_padded(_u32(am_ptr)), am_ent=_padded(_u32(am_ent)), gm_ptr=_u32(gm_ptr),
        gm_agent=gm_agent.contiguous(), pc=pc.contiguous(), cls=_padded(cls.contiguous(), 64), small_groups=_u32(small),
        chunk_group=_u32(chunk_group), chunk_begin=_u32(chunk_begin), chunk_end=_u32(chunk_end),
        chunk_part=chunk_part.to(torch.int32), big_groups=_u32(big_groups), big_part_ptr=_u32(big_part_ptr),
        n_parts=n_parts, tile_begin=_padded(_u32(tile_begin), 4), tile_flags=_padded(_u32(tile_flags), 4),
        ent1=_padded(_u32(ent1)), device=dev,
        orig_id=None if orig_id is None else _padded(_u32(orig_id.to(dev))),
        n_giant_chunks=n_giant_chunks, n_giant_big=n_giant_big,
    )


class NativeWorld:
    """A world built by ``gj_world_build`` (the C-ABI builder, csrc/gj_world.cu) from the reference's arrays of
    ``data``: the handle owns the device arrays; ``desc()`` is what the step entry points take.  ``host=True`` runs
    the same build on the CPU (``gj_world_build_host``; its arrays then live in host memory — for comparing with
    :func:`build_csr` in the CPU tests, never for stepping)."""

    def __init__(self, data: "HeteroData", device="cuda:0", renumber=True, host=False, want_tiers=None):
        import ctypes as C

        from . import _lib
        L = _lib.lib()
        dev = torch.device("cpu" if host else device)
        types = data.venue_types()
        src = _lib.WorldSrc()
        keep = []

        def ptr(t, dtype):
            t = torch.as_tensor(t).to(device=dev, dtype=dtype).contiguous()
            keep.append(t)
            return t.data_ptr()

        n = len(data["agent"].id)
        src.n_agents, src.n_types, src.renumber = n, len(types), 1 if renumber else 0
        for i, t in enumerate(types):
            ei = data["attends_" + t].edge_index
            src.type_name[i] = t.encode()
            src.edge_agent[i], src.edge_group[i] = ptr(ei[0], torch.long), ptr(ei[1], torch.long)
            src.n_edges[i], src.n_groups[i] = ei.shape[1], len(data[t]["id"])
            people = torch.as_tensor(data[t]["people"])
            if people.dtype.is_floating_point:
                src.people_f32[i] = ptr(people, torch.float32)
            else:
                src.people_i64[i] = ptr(people, torch.long)
        src.age, src.sex = ptr(data["agent"].age, torch.long), ptr(data["agent"].sex, torch.long)
        if "original_index" in data["agent"]:
            src.original_index = ptr(data["agent"]["original_index"], torch.long)
        if want_tiers is not None:
            src.want_tier = ptr(torch.tensor([int(want_tiers.get(t, TIER_GENERIC)) for t in types]), torch.int32)
        handle = C.c_void_p()
        ctx = torch.cuda.device(dev) if dev.type == "cuda" else _NullContext()
        with ctx:
            rc = (L.gj_world_build_host if host else L.gj_world_build)(C.byref(src), C.byref(handle))
        if rc != 0:
            raise _lib.GradJuneLibraryError(f"gj_world_build failed ({rc}): {L.gj_world_last_error().decode()}")
        self._lib, self.handle, self.device, self.host, self.types, self.n_agents = L, handle, dev, host, types, n
        self._desc = L.gj_world_descriptor(handle).contents
        # what grad_june.ops / partition read from a world object (so that a native world can be stepped like a
        # DeviceWorld: get_device_world(..., native=True))
        d = self._desc
        self.n_groups, self.n_edges = int(d.n_groups), int(d.n_edges)
        self.type_group_off = [int(d.type_group_off[i]) for i in range(len(types) + 1)]
        self.type_tier = [int(d.type_tier[i]) for i in range(len(types))]
        self.orig_id = self.array("orig_id", n) if d.orig_id else None

    def desc(self):
        return self._desc

    @property
    def dbeta_w(self):
        return self.__dict__.get("_dbeta_w")

    @dbeta_w.setter
    def dbeta_w(self, t):       # partitioned worlds: the per-group ownership weights live with the caller
        self.__dict__["_dbeta_w"] = t
        self._desc.dbeta_w = t.data_ptr()

    def permutation(self):
        """perm[new] = old of the renumbering the build applied (int64 tensor on the build's device), None = identity."""
        p = self._lib.gj_world_permutation(self.handle)
        if not p:
            return None
        return self._view(p, self.n_agents, torch.long)

    def _view(self, address, count, dtype):
        """Copy of ``count`` elements at ``address`` (host or device memory of the handle) as a tensor."""
        import ctypes as C
        out = torch.empty(count, dtype=dtype)
        nbytes = out.numel() * out.element_size()
        if self.host:
            C.memmove(out.data_ptr(), address, nbytes)
            return out
        out = out.to(self.device)
        from . import _lib
        with torch.cuda.device(self.device):
            _lib.check(self._lib.gj_memcpy(out.data_ptr(), address, nbytes), "gj_memcpy")
        return out

    def array(self, name, count, dtype=torch.int32, index=None):
        """Copy of one descriptor array (``index``: the edge type of a per-type array)."""
        field = getattr(self._desc, name)
        address = field[index] if index is not None else field
        if not address or count == 0:
            return torch.zeros(0, dtype=dtype)
        return self._view(address, count, dtype)

    def close(self):
        if self.handle:
            self._lib.gj_world_destroy(self.handle)
            self.handle = None

    def __del__(self):
        if sys is None or sys.is_finalizing():   # the CUDA context may already be gone: leave it to process teardown
            return
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


class _NullContext:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def get_device_world(data: HeteroData, device, small_group: Optional[int] = None, chunk: Optional[int] = None,
                     native: Optional[bool] = None):
    """CSR layout of ``data`` on ``device``; cached on the world object and rebuilt when an edge list,
    ``people`` or the agent attributes are replaced (identity + version check).  ``native`` (default: the
    environment variable GJ_NATIVE_BUILD=1): build it with the C-ABI builder ``gj_world_build`` instead of the torch
    code below (identical arrays, tests/test_world_build.py)."""
    import os
    if native is None:
        native = os.environ.get("GJ_NATIVE_BUILD", "0") == "1"
    cache = data.__dict__.setdefault("_gj_cache", {})
    if cache.get("frozen") == str(device):
        return cache["world"]
    types = data.venue_types()
    sig = [str(device)]
    for t in types:
        ei = data["attends_" + t].edge_index
        pp = data[t]["people"]
        sig.append((t, id(ei), ei._version, tuple(ei.shape), id(pp), getattr(pp, "_version", 0), len(data[t]["id"])))
    oi = data["agent"]["original_index"] if "original_index" in data["agent"] else None
    sig.append((id(data["agent"].age), id(data["agent"].sex), id(oi)))
    sig = tuple(sig)
    if cache.get("sig") == sig:
        return cache["world"]
    if small_group is None or chunk is None:
        from . import _lib

        cfg = _lib.config()
        small_group, chunk = cfg["small_group"], cfg["chunk"]
    n = len(data["agent"].id)
    if native and torch.device(device).type == "cuda":
        world = NativeWorld(data, device=device, renumber=False, want_tiers=agreed_tiers(data, device))
        cache["sig"] = sig
        cache["world"] = world
        cache.pop("scratch", None)
        return world
    world = build_csr(
        n, types,
        {t: data["attends_" + t].edge_index for t in types},
        {t: torch.as_tensor(data[t]["people"]) for t in types},
        {t: len(data[t]["id"]) for t in types},
        torch.as_tensor(data["agent"].age), torch.as_tensor(data["agent"].sex), small_group, chunk, device,
        orig_id=None if oi is None else torch.as_tensor(oi), want_tiers=agreed_tiers(data, device),
    )
    cache["sig"] = sig
    cache["world"] = world
    cache.pop("scratch", None)
    return world


def agreed_tiers(data: HeteroData, device):
    """None for an ordinary world.  For one part of a geographically partitioned world: the layout tier every
    rank will use per edge type (ADVICE r1: tiers chosen from the local slice alone can differ between ranks, and
    then the packed boundary buffers they all-reduce have different layouts).  Each rank tries its tiers locally;
    a type keeps a streaming tier only if EVERY rank achieved it and — for the RANGE tier, which has no per-group
    buffer to exchange — no group of the type straddles partitions.  Collective: every rank calls it at its first
    step."""
    part = data.__dict__.get("_gj_partition")
    if part is None or part.world_size == 1:
        return None
    import torch.distributed as dist

    types = data.venue_types()
    n = len(data["agent"].id)
    edges = {t: data["attends_" + t].edge_index.to(device) for t in types}
    n_groups = {t: len(data[t]["id"]) for t in types}
    range_type, cell_type = tier_candidates(n, types, edges, n_groups)
    mine = torch.zeros(len(types), dtype=torch.long)
    for ti, t in enumerate(types):
        ei = edges[t]
        if t == range_type and part.n_boundary.get(t, 0) == 0:
            pc = p_contact(torch.as_tensor(data[t]["people"]).to(device))
            if _try_range_tier(n, ei[0], ei[1], n_groups[t], pc) is not None:
                mine[ti] = TIER_RANGE
        elif t == cell_type and _try_cell_tier(n, ei[0], ei[1], n_groups[t]) is not None:
            mine[ti] = TIER_CELL
    backend = dist.get_backend(part.process_group)
    buf = mine.to(device) if backend == "nccl" else mine
    both = torch.stack((buf, -buf))
    dist.all_reduce(both, op=dist.ReduceOp.MIN, group=part.process_group)
    lo, hi = both[0].cpu(), (-both[1]).cpu()
    return {t: (int(lo[ti]) if int(lo[ti]) == int(hi[ti]) else TIER_GENERIC) for ti, t in enumerate(types)}


def freeze_device_world(data: HeteroData, device, drop_edge_lists: bool = True):
    """Build the CSR layout once and pin it: later calls return it without looking at the edge lists,
    which can then be dropped (an England-scale world's int64 [2,E] lists are ~4 GB the kernels never read)."""
    world = get_device_world(data, device)
    data._gj_cache["frozen"] = str(device)
    if drop_edge_lists:
        for key in list(data._edge_store_dict):
            store = data._edge_store_dict[key]
            if "edge_index" in store:
                store.edge_index = store.edge_index[:, :0]
    return world


# --------------------------------------------------------------------------------------
# synthetic worlds
# --------------------------------------------------------------------------------------
def create_simple_connected_graph(n_agents, device="cpu", params=None):
    """BASELINE config 1 world (reference utils.py:97-133): even agents share one household, odd
    agents one school, ``people = n_agents`` for both, uniform ages and sexes."""
    from .transmission import TransmissionSampler

    data = HeteroData()
    sampler = TransmissionSampler.from_file() if params is None else TransmissionSampler.from_parameters(params)
    ids = torch.arange(0, n_agents)
    data["agent"].id = ids
    data["agent"].age = torch.randint(0, 100, (n_agents,))
    data["agent"].sex = torch.randint(0, 2, (n_agents,))
    values = sampler(n_agents)
    data["agent"].infection_parameters = {
        k: values[i] for i, k in enumerate(("max_infectiousness", "shape", "rate", "shift"))
    }
    data["agent"].transmission = torch.zeros(n_agents)
    data["agent"].susceptibility = torch.ones(n_agents)
    data["agent"].is_infected = torch.zeros(n_agents)
    data["agent"].infection_time = torch.zeros(n_agents)
    data["agent"].symptoms = {
        "current_stage": torch.ones(n_agents, dtype=torch.long),
        "next_stage": torch.ones(n_agents, dtype=torch.long),
        "time_to_next_stage": torch.zeros(n_agents),
    }
    data["agent"].ethnicity = np.array(["A"] * n_agents)
    for name, members in (("household", ids[::2]), ("school", ids[1::2])):
        data[name].id = torch.zeros(1)
        data[name].people = torch.tensor([n_agents])
        data["agent", "attends_" + name, name].edge_index = torch.vstack(
            (members, torch.zeros(members.numel(), dtype=torch.long)))
    data = ToUndirected()(data)
    return data.to(device)


_HOUSEHOLD_SIZES = torch.tensor([1, 2, 3, 4, 5, 6, 8])
_HOUSEHOLD_PROBS = torch.tensor([0.41, 0.33, 0.11, 0.09, 0.03, 0.025, 0.005])


def _company_table(n_agents, n_sa, seed, block, device):
    """Companies of one block of the synthetic world: log-normal sizes (clipped to [1, 5000]), home super-area
    uniform inside the block and sorted.  A function of (seed, block) alone, so every rank of a partitioned
    world can rebuild the tables of its neighbours."""
    g = torch.Generator(device=device)
    g.manual_seed(int(seed) * 1_000_003 + 7919 * int(block) + 17)
    n_comp = max(n_agents // 25, 1)
    csize = torch.exp(1.5 + 1.3 * torch.randn(n_comp, generator=g, device=device)).clamp(1, 5000)
    chome = torch.sort(torch.randint(0, n_sa, (n_comp,), generator=g, device=device))[0]
    return csize, chome


def make_synthetic_world(n_agents: int, seed: int = 0, device="cpu", agents_per_super_area: int = 7500,
                         with_reverse: bool = False, block=None, super_areas_per_region: int = 1000) -> HeteroData:
    """England-like synthetic world (SURVEY.md §8d, config 3): area-contiguous agents, contiguous
    households (1-8 members), schools (ages 5-17, two per super-area), universities (18-22),
    companies (19-64, log-normal sizes, 80 % in the home super-area, 20 % uniform over the home region of
    ``super_areas_per_region`` super-areas), care homes (over 75 + staff) and three leisure groups per agent (own
    super-area and the two neighbouring ones).  ``people`` = member count.
    Generated with torch ops on ``device`` so the 56 M-agent world builds on the GPU in seconds.

    ``block=(b, B)``: generate only block ``b`` of a world made of ``B`` such blocks of ``n_agents`` agents each
    (one block per GPU of a geographically partitioned run; no rank ever holds the whole world).  Agent indices are
    local to the block, group ids are GLOBAL (``data[t].n_global`` groups; ``data[t].scope`` says whether other
    blocks can attend them), ``people`` counts only this block's members:
    :func:`grad_june.partition.partition_from_blocks` turns this into the rank's local world."""
    dev = torch.device(device)
    b, B = (0, 1) if block is None else (int(block[0]), int(block[1]))
    g = torch.Generator(device=dev)
    g.manual_seed(seed + 7919 * b)
    N = int(n_agents)
    SA = agents_per_super_area
    ids = torch.arange(N, device=dev)
    n_sa = int((N + SA - 1) // SA)           # super-areas per block
    n_sa_g = n_sa * B                        # ... of the whole world
    sa = ids // SA + b * n_sa                # global super-area of each agent

    def rand(n):
        return torch.rand(n, generator=g, device=dev)

    # age pyramid: flat to 60, then linearly thinning to 99
    w_age = torch.ones(100, device=dev)
    w_age[60:] = torch.linspace(1.0, 0.05, 40, device=dev)
    age = torch.multinomial(w_age, N, replacement=True, generator=g)
    sex = (rand(N) < 0.5).long()

    data = HeteroData()
    data["agent"].id = ids
    data["agent"].age = age
    data["agent"].sex = sex

    def add(name, agents, groups, n_groups, scope="global"):
        data[name].id = torch.arange(n_groups, device=dev) if block is None else torch.zeros(0, device=dev)
        if block is None:
            data[name].people = torch.bincount(groups, minlength=n_groups)
        else:
            data[name].n_global, data[name].scope = int(n_groups), scope
        data["agent", "attends_" + name, name].edge_index = torch.stack((agents, groups))

    # households: contiguous runs of agents, never shared between blocks (ids local to the block)
    m = max(N // 2, 1) + 16
    hs = _HOUSEHOLD_SIZES.to(dev)[torch.multinomial(_HOUSEHOLD_PROBS.to(dev), m, replacement=True, generator=g)]
    ends = torch.cumsum(hs, 0)
    n_hh = int(torch.searchsorted(ends, torch.tensor([N], device=dev), right=False)[0]) + 1
    hh = torch.searchsorted(ends[:n_hh].contiguous(), ids, right=True)
    add("household", ids, hh, n_hh, scope="local")

    r = rand(N)
    is_school = (age >= 5) & (age <= 17)
    is_uni = (age >= 18) & (age <= 22) & (r < 0.3)
    adult = (age >= 19) & (age <= 64) & ~is_uni
    is_care_worker = adult & (r > 0.998)
    is_worker = adult & (r < 0.75) & ~is_care_worker
    is_resident = (age > 75) & (r < 0.04)

    a = ids[is_school]
    add("school", a, sa[a] * 2 + (rand(a.numel()) < 0.5).long(), n_sa_g * 2)
    a = ids[is_uni]
    n_uni = max(n_sa_g // 111, 1)
    add("university", a, torch.clamp(sa[a] // 111, max=n_uni - 1), n_uni)

    # companies: log-normal sizes, home super-area uniform; workers pick proportionally to size, 80 % among the
    # companies of their own super-area, 20 % among those of their region
    a = ids[is_worker]
    tables = [_company_table(N, n_sa, seed, j, dev) for j in range(B)]
    csize = torch.cat([t[0] for t in tables])
    chome = torch.cat([t[1] + j * n_sa for j, t in enumerate(tables)])     # ascending: blocks are in order
    n_comp = csize.numel()
    cum = torch.cumsum(csize.double(), 0)
    cum0 = torch.cat((torch.zeros(1, dtype=cum.dtype, device=dev), cum))
    first = torch.searchsorted(chome, torch.arange(n_sa_g + 1, device=dev))   # companies of each super-area
    RS = max(int(super_areas_per_region), 1)
    sa_a = sa[a]
    lo, hi = cum0[first[sa_a]], cum0[first[sa_a + 1]]
    reg_lo = (sa_a // RS) * RS
    reg_hi = torch.clamp(reg_lo + RS, max=n_sa_g)
    rlo, rhi = cum0[first[reg_lo]], cum0[first[reg_hi]]
    u = rand(a.numel()).double()
    local = (rand(a.numel()) < 0.8) & (hi > lo)
    target = torch.where(local, lo + u * (hi - lo), rlo + u * (rhi - rlo))
    comp = torch.searchsorted(cum, target, right=True).clamp(max=n_comp - 1)
    add("company", a, comp, n_comp)

    a = torch.cat((ids[is_resident], ids[is_care_worker]))
    add("care_home", a, sa[a], n_sa_g)

    # leisure: own super-area and its two neighbours (k = 3 nearest, graph_loader.py:12)
    left = torch.where(sa == 0, torch.full_like(sa, min(2, n_sa_g - 1)), sa - 1)
    right = torch.where(sa == n_sa_g - 1, torch.full_like(sa, max(n_sa_g - 3, 0)), sa + 1)
    if n_sa_g >= 3:
        la = torch.cat((ids, ids, ids))
        lg = torch.cat((sa, left, right))
    else:
        la, lg = ids, sa
    add("leisure", la, lg, n_sa_g)
    data["agent"].ethnicity = np.array(["A"])  # one label; per-agent strings are not needed by the step
    if block is not None:
        data.__dict__["_gj_block"] = (b, B, N)
    elif with_reverse:
        data = ToUndirected()(data)
    return data
