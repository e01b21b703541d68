"""gj_world_build (csrc/gj_world.cu: the world builder behind the C ABI, Thrust/CUB) against the Python builder
(grad_june/world.py): the HOST instantiation of the same code (gj_world_build_host) must produce, array for array,
what layout_order + build_csr produce — on the reference's sample world as loaded (households scattered: it
renumbers), on a synthetic world loaded shuffled, and on BASELINE config 1's two-giant-groups world."""
import numpy as np
import pytest
import torch

import helpers as H
from grad_june import world as W


def _python_build(data):
    types = data.venue_types()
    n = len(data["agent"].id)
    return W.build_csr(n, types, {t: data["attends_" + t].edge_index for t in types},
                       {t: torch.as_tensor(data[t]["people"]) for t in types}, {t: len(data[t]["id"]) for t in types},
                       data["agent"].age, data["agent"].sex, 16, 1024, "cpu",
                       orig_id=data["agent"]["original_index"] if "original_index" in data["agent"] else None)


def _compare(native, ref, types):
    d = native.desc()
    n, G = ref.n_agents, ref.n_groups
    assert (d.n_agents, d.n_groups, d.n_edges, d.n_types) == (n, G, ref.n_edges, len(types))
    assert list(d.type_group_off[:len(types) + 1]) == list(ref.type_group_off)
    assert list(d.type_tier[:len(types)]) == list(ref.type_tier)
    assert (d.n_small, d.n_chunks, d.n_big, d.n_parts) == (ref.small_groups.numel(), ref.chunk_group.numel(),
                                                           ref.big_groups.numel(), ref.n_parts)
    assert (d.n_giant_chunks, d.n_giant_big) == (ref.n_giant_chunks, ref.n_giant_big)
    assert d.n_tiles == ref.tile_begin.numel() - 1
    E = ref.n_generic_edges
    for name, count in (("am_ptr", n + 1), ("am_ent", E), ("gm_ptr", G + 1), ("gm_agent", E), ("small_groups", d.n_small),
                        ("chunk_group", d.n_chunks), ("chunk_begin", d.n_chunks), ("chunk_end", d.n_chunks),
                        ("chunk_part", d.n_chunks), ("big_groups", d.n_big), ("big_part_ptr", d.n_big + 1),
                        ("tile_begin", d.n_tiles + 1), ("tile_flags", d.n_tiles), ("ent1", n)):
        mine = native.array(name, count)
        assert torch.equal(mine, getattr(ref, name)[:count].cpu().to(torch.int32)), name
    assert torch.equal(native.array("pc", G, torch.float32), ref.pc.cpu())
    assert torch.equal(native.array("cls", n, torch.uint8), ref.cls[:n].cpu())
    if ref.orig_id is not None:
        assert torch.equal(native.array("orig_id", n), ref.orig_id[:n].cpu())
    else:
        assert not d.orig_id
    cells_total = 0
    for ti, t in enumerate(types):
        if ref.type_tier[ti] == W.TIER_RANGE:
            assert bool(d.range_pc_from_size[ti]) == bool(ref.range_pc_from_size[ti]), t
            assert torch.equal(native.array("range_slot", n, index=ti), ref.range_slot[ti][:n].cpu()), t
            assert torch.equal(native.array("range_pc", n, torch.float32, index=ti), ref.range_pc[ti][:n].cpu()), t
        elif ref.type_tier[ti] == W.TIER_CELL:
            c = ref.cells[ti]
            Gt = ref.type_group_off[ti + 1] - ref.type_group_off[ti]
            assert d.n_cells[ti] == c["n_cells"] and d.cell_off[ti] == cells_total
            for name, count in (("tile_cell", d.n_tiles), ("cell_tile_ptr", c["n_cells"] + 1),
                                ("cell_grp_ptr", c["n_cells"] + 1), ("cell_grp", c["cell_grp"].numel()),
                                ("grp_cell_ptr", Gt + 1), ("grp_cell", c["grp_cell"].numel())):
                assert torch.equal(native.array(name, count, index=ti), c[name].cpu().to(torch.int32)), (t, name)
            cells_total += c["n_cells"]
    assert d.n_cells_total == cells_total


def test_native_build_of_the_sample_world_matches_python(golden_dir):
    data = W.world_from_arrays(np.load(golden_dir / "sample_world.npz"), H.SAMPLE_TYPES)
    native = W.NativeWorld(data, host=True, renumber=True)
    perm = native.permutation()
    data = W.renumber_world(data)
    assert perm is not None and torch.equal(perm, data["agent"].original_index)
    ref = _python_build(data)
    hi = data.venue_types().index("household")
    assert ref.type_tier[hi] == W.TIER_RANGE and ref.range_pc_from_size[hi]
    _compare(native, ref, data.venue_types())
    native.close()


def test_native_build_without_renumbering_keeps_the_loaded_numbering(golden_dir):
    data = W.world_from_arrays(np.load(golden_dir / "sample_world.npz"), H.SAMPLE_TYPES)
    native = W.NativeWorld(data, host=True, renumber=False)
    assert native.permutation() is None
    ref = _python_build(data)
    assert ref.type_tier[data.venue_types().index("household")] == W.TIER_GENERIC
    _compare(native, ref, data.venue_types())


def test_native_build_of_a_shuffled_synthetic_world():
    n = 30_000
    data = W.make_synthetic_world(n, seed=7, agents_per_super_area=2500)
    laid_out = W.NativeWorld(data, host=True)
    assert laid_out.permutation() is None           # already laid out: nothing to renumber
    _compare(laid_out, _python_build(data), data.venue_types())
    data = W.renumber_world(data, torch.randperm(n, generator=torch.Generator().manual_seed(3)))
    native = W.NativeWorld(data, host=True)         # carries original_index in: the build composes it
    perm = native.permutation()
    data = W.renumber_world(data)
    assert torch.equal(data["agent"].original_index, torch.arange(n))
    ref = _python_build(data)
    assert ref.range_pc_from_size[data.venue_types().index("household")]
    _compare(native, ref, data.venue_types())
    assert perm is not None


def test_native_build_of_config1_world_with_giant_groups():
    n = 80_000                                      # two groups of 40 000 members: giant (> GJ_SCATTER_MAX_GROUP)
    torch.manual_seed(0)
    data = W.create_simple_connected_graph(n)
    native = W.NativeWorld(data, host=True)
    ref = _python_build(data)
    assert ref.n_giant_big == 2 and ref.n_giant_chunks == 80
    _compare(native, ref, data.venue_types())


def test_native_build_rejects_bad_indices():
    from grad_june import _lib
    data = W.make_synthetic_world(2000, seed=1, agents_per_super_area=500)
    ei = data["attends_company"].edge_index.clone()
    ei[0, 0] = 5000
    data["attends_company"].edge_index = ei
    with pytest.raises(_lib.GradJuneLibraryError, match="agent index out of range"):
        W.NativeWorld(data, host=True)
