"""JUNE world (HDF5) -> the world container the step runs on (reference: grad_june/june_world_loader/*.py,
example_scripts/make_data.py).

The reference builds its edge lists with Python loops over every person (network_loader.py:14-25,30-44) and one
BallTree query + ``torch.hstack`` per super-area (leisure_loader.py:38-73): minutes for a city, not feasible for
England.  Here the same edge lists — same edges, same ORDER (the order fixes the reference's summation order) — come
from a handful of vectorised numpy passes.  The arrays are taken from any mapping with the JUNE file's layout
(``population/{id,age,sex,ethnicity,area,super_area,group_ids,group_specs}``, ``geography/{area_name,
area_socioeconomic_indices,super_area_coordinates,super_area_id}``, ``<venues>/id``): an open ``h5py.File`` when h5py
is installed (:func:`load_june_world`), or plain dicts of numpy arrays (tests, other containers).

The result is a :class:`grad_june.world.HeteroData` with the reference's node / edge stores; ``Runner.get_data``
renumbers it (``world.renumber_world``) so that the streaming layout tiers apply.
"""
from typing import Mapping, Sequence

import numpy as np
import torch

from .world import HeteroData, ToUndirected

# spec -> (plural = HDF5 group holding the venue ids, columns of population/group_ids searched)   [*_loader.py]
NETWORK_SPECS = {
    "household": ("households", (0,)),
    "care_home": ("care_homes", (0, 1)),
    "company": ("companies", (1,)),
    "school": ("schools", (1,)),
    "university": ("universities", (1,)),
}
LOAD_ORDER = ("household", "care_home", "company", "school", "university")     # graph_loader.py:20-26


def _as_str(a):
    a = np.asarray(a)
    return a.astype("U") if a.dtype.kind in "SO" else a


def network_edges(group_ids: np.ndarray, group_specs: np.ndarray, spec: str, columns: Sequence[int]):
    """(person, group) of every membership of venue type ``spec``, in the reference's edge order:
    network_loader.py:14-25 scans the columns in turn and the persons in ascending order, appending person i to
    ``ret[group_id]``; network_loader.py:33-37 then emits the groups in the order they were FIRST seen and each
    group's members in append order.  Also returns the member count per group id seen."""
    group_ids = np.asarray(group_ids)
    specs = _as_str(group_specs)
    persons, gids = [], []
    for c in columns:
        hit = np.nonzero(specs[:, c] == spec)[0]
        persons.append(hit)
        gids.append(group_ids[hit, c])
    persons = np.concatenate(persons) if persons else np.zeros(0, dtype=np.int64)
    gids = np.concatenate(gids).astype(np.int64) if gids else np.zeros(0, dtype=np.int64)
    if gids.size == 0:
        return persons.astype(np.int64), gids, {}
    uniq, first, inverse, counts = np.unique(gids, return_index=True, return_inverse=True, return_counts=True)
    rank_of_group = np.empty(uniq.size, dtype=np.int64)
    rank_of_group[np.argsort(first, kind="stable")] = np.arange(uniq.size)      # first-seen order of the groups
    order = np.argsort(rank_of_group[inverse], kind="stable")                   # members keep their append order
    return persons[order].astype(np.int64), gids[order], dict(zip(uniq.tolist(), counts.tolist()))


def leisure_edges(person_super_area: np.ndarray, super_area_ids: np.ndarray, coordinates_deg: np.ndarray, k: int):
    """Leisure edges (leisure_loader.py:38-73): every super-area is one leisure group attended by all residents of
    its k nearest super-areas (haversine BallTree over the coordinates in radians, itself included), emitted group
    by group in ``super_area_ids`` order, the neighbours in query order, residents in ascending person order."""
    from sklearn.neighbors import BallTree

    person_sa = np.asarray(person_super_area).astype(np.int64)
    ids = np.asarray(super_area_ids).astype(np.int64)
    coords = np.deg2rad(np.asarray(coordinates_deg, dtype=np.float64))
    tree = BallTree(coords, metric="haversine")
    # the reference indexes the coordinate table by the super-area ID itself (leisure_loader.py:47-49)
    _, near = tree.query(coords[ids], k=k)                                     # [S, k] neighbour super-areas
    by_sa = np.argsort(person_sa, kind="stable")                                # residents of each super-area, ascending
    n_sa = int(max(person_sa.max(initial=-1), near.max(initial=-1), ids.max(initial=-1))) + 1
    count = np.bincount(person_sa, minlength=n_sa)
    start = np.concatenate(([0], np.cumsum(count)))
    seg_sa = near.reshape(-1)                                                   # (group, neighbour) pairs in emit order
    seg_len = count[seg_sa]
    seg_off = np.concatenate(([0], np.cumsum(seg_len)))
    total = int(seg_off[-1])
    seg = np.repeat(np.arange(seg_sa.size), seg_len)
    people = by_sa[start[seg_sa][seg] + (np.arange(total) - seg_off[:-1][seg])]
    groups = np.repeat(ids, seg_len.reshape(len(ids), k).sum(1))
    return people.astype(np.int64), groups.astype(np.int64), seg_len.reshape(len(ids), k).sum(1).astype(np.int64)


def world_from_june_arrays(f: Mapping, k_leisure: int = 3, load_leisure: bool = True,
                           specs: Sequence[str] = LOAD_ORDER) -> HeteroData:
    """GraphLoader.load_graph + AgentDataLoader.load_agent_data (graph_loader.py:16-39, agent_data_loader.py:20-33)
    from a mapping with the JUNE file's layout."""
    pop, geo = f["population"], f["geography"]
    data = HeteroData()
    group_ids = np.asarray(pop["group_ids"][:])
    group_specs = pop["group_specs"][:]
    for spec in specs:
        plural, columns = NETWORK_SPECS[spec]
        person, group, counts = network_edges(group_ids, group_specs, spec, columns)
        ids = np.asarray(f[plural]["id"][:])
        data[spec].id = ids
        data[spec].people = torch.tensor([counts.get(int(i), 0) for i in ids], dtype=torch.long)   # network_loader.py:39-41
        data["agent", "attends_" + spec, spec].edge_index = torch.from_numpy(np.vstack((person, group)))
    if load_leisure:
        sa_ids = np.asarray(geo["super_area_id"][:])
        person, group, people = leisure_edges(pop["super_area"][:], sa_ids, geo["super_area_coordinates"][:], k_leisure)
        data["agent", "attends_leisure", "leisure"].edge_index = torch.from_numpy(np.vstack((person, group)))
        data["leisure"].id = torch.from_numpy(sa_ids.astype(np.int64))
        data["leisure"].people = torch.from_numpy(people)
    data = ToUndirected()(data)
    # agent attributes (agent_data_loader.py:20-33)
    agent = data["agent"]
    agent.id = torch.as_tensor(np.asarray(pop["id"][:]))
    agent.age = torch.as_tensor(np.asarray(pop["age"][:]).astype(np.int64))
    agent.ethnicity = _as_str(pop["ethnicity"][:])
    area_ids = np.asarray(pop["area"][:])
    bins = [0, 0.20, 0.4, 0.6, 0.8, 1.0]
    agent.socioeconomic_index = torch.as_tensor(
        np.digitize(np.asarray(geo["area_socioeconomic_indices"][:])[area_ids], bins), dtype=torch.int8)
    agent.area = _as_str(np.asarray(geo["area_name"][:])[area_ids])
    agent.super_area = torch.as_tensor(np.asarray(pop["super_area"][:]).astype(np.int64))   # results_by: super_area
    sexes = _as_str(pop["sex"][:])
    agent.sex = torch.as_tensor((sexes == "f").astype(np.int64))                # "m" -> 0, "f" -> 1
    return data


def load_june_world(june_world_path, k_leisure: int = 3, load_leisure: bool = True) -> HeteroData:
    """example_scripts/make_data.py for a JUNE HDF5 world file.  Needs h5py (not part of this image: the function
    raises ImportError with that explanation; everything it calls is exercised on plain arrays by the tests)."""
    try:
        import h5py
    except ImportError as e:  # pragma: no cover
        raise ImportError("reading a JUNE world file needs h5py; world_from_june_arrays() takes the same layout as "
                          "plain numpy arrays") from e
    with h5py.File(june_world_path, "r") as f:
        return world_from_june_arrays(f, k_leisure=k_leisure, load_leisure=load_leisure)


class GraphLoader:
    """The reference's loader class (graph_loader.py:10-39) over the vectorised functions above."""

    def __init__(self, june_world_path, k_leisure=3):
        self.june_world_path = june_world_path
        self.k_leisure = k_leisure

    def load_graph(self, data=None, load_leisure=True):
        return load_june_world(self.june_world_path, self.k_leisure, load_leisure)
