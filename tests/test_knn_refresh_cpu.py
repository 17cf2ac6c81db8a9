"""CPU: the one-pass layout rules of grl_knn_topology (tests/knn_topology_reference.py) against the long way round
(oracle.graph.knn_edges + coalesce, stable counting sorts of both CSRs, the gathers of a fixed-capacity set), and when the
data builders rebuild kNN edges in place (`knn_in_place`)."""
import itertools

import numpy as np
import pytest
import torch

from geometry_rl_b200.synthetic import CONFIGS, observation_layout
from tests.knn_topology_reference import chain_layouts, neighbour_lists, one_pass_layouts

FIELDS = ("coo", "edge_ptr", "rowptr_dst", "edge_src", "edge_dst", "eid_coo", "rowptr_src", "src_eid", "s_src", "s_dst")


def _cases():
    rng = np.random.default_rng(7)
    out = []
    P = 11
    pos = rng.standard_normal((7, P, 3)).astype(np.float32)
    # num_valid 0, 1, 2, <= k, P and in between; the first graph has no edge, so the tails come from graph 2
    out.append(("ragged", pos, np.array([1, 0, 2, 3, P, 7, 4], np.int32), 3))
    out.append(("all_valid", pos, None, 3))
    out.append(("k_equals_P_minus_1", rng.standard_normal((3, 9, 3)).astype(np.float32), np.array([9, 5, 9], np.int32), 8))
    # a 3x3x3 lattice: many equal distances, ties go to the lower index
    g = np.stack(np.meshgrid(np.arange(3.0), np.arange(3.0), np.arange(3.0), indexing="ij"), -1).reshape(-1, 3)
    out.append(("lattice_ties", np.broadcast_to(g * 0.5, (2, 27, 3)).astype(np.float32).copy(),
                np.array([27, 20], np.int32), 4))
    # no edge anywhere: every tail entry is 0
    out.append(("all_empty", pos[:3], np.array([0, 1, 1], np.int32), 3))
    # non-finite points: NaN distances rank as +inf, ties by index
    bad = rng.standard_normal((5, P, 3)).astype(np.float32)
    bad[0, 3, 1] = np.nan
    bad[1, :, :] = np.nan
    bad[2, 0] = np.inf
    bad[2, 5, 2] = -np.inf
    bad[3, 2] = 1e30  # finite, but its squared distances overflow to +inf
    out.append(("non_finite", bad, np.array([P, 6, P, 9, 2], np.int32), 3))
    return out


def _capacities(pos, nv, k):
    B, P, _ = pos.shape
    exact = B * P * max(0, min(k, P - 1))
    return ([exact] if nv is None else []) + [B * P * k]


@pytest.mark.parametrize("case", range(6))
def test_one_pass_rules_equal_the_long_way(case):
    name, pos, nv, k = _cases()[case]
    for cap in _capacities(pos, nv, k):
        a, b = one_pass_layouts(pos, nv, k, cap), chain_layouts(pos, nv, k, cap)
        for f in FIELDS:
            assert a[f].dtype == b[f].dtype and a[f].shape == b[f].shape, (name, cap, f)
            assert np.array_equal(a[f], b[f]), (name, cap, f)
        B, P, _ = pos.shape
        E = int(a["edge_ptr"][-1])
        for f in ("edge_src", "edge_dst", "s_src", "s_dst"):
            assert a[f].min(initial=0) >= 0 and a[f].max(initial=0) < B * P, (name, f)  # in bounds, NaNs included
        for f in ("eid_coo", "src_eid"):
            assert a[f].max(initial=0) < max(E, 1), (name, f)
        assert sorted(a["eid_coo"][:E]) == list(range(E)) and sorted(a["src_eid"][:E]) == list(range(E))


@pytest.mark.parametrize("case", [0, 1, 2, 3, 4])
def test_neighbour_lists_equal_the_oracle_knn_for_finite_points(case):
    from oracle import graph as og
    name, pos, nv, k = _cases()[case]
    B, P, _ = pos.shape
    for g in range(B):
        pv = P if nv is None else int(nv[g])
        lists = neighbour_lists(pos[g, :pv], k)
        mine = og.coalesce(torch.tensor([[j for lst in lists for j in lst],
                                         [i for i, lst in enumerate(lists) for _ in lst]], dtype=torch.long).reshape(2, -1))
        assert torch.equal(mine, og.knn_edges(torch.from_numpy(pos[g, :pv]), k)), (name, g)


def test_non_finite_points_get_exactly_k_neighbours():
    _, pos, nv, k = _cases()[5]
    lists = neighbour_lists(pos[1, :6], k)  # every distance NaN: the k lowest other indices
    assert lists == [[1, 2, 3], [0, 2, 3], [0, 1, 3], [0, 1, 2], [0, 1, 2], [0, 1, 2]]
    lists = neighbour_lists(pos[0], k)
    assert all(len(lst) == k and 3 not in lst for i, lst in enumerate(lists) if i != 3)  # NaN point ranks last
    assert lists[3] == [0, 1, 2]


def _data(task, **kw):
    if task == "rope":
        from geometry_rl_b200.modules.pyg_data.rope_tasks_data import RopeTasksData as D
        cfg = CONFIGS["rope_shaping_hepi_trpl_cfg"]
    else:
        from geometry_rl_b200.modules.pyg_data.rigid_tasks_data import RigidTasksData as D
        cfg = CONFIGS["rigid_insertion_multi_hepi_trpl_cfg"]
    dims, names = observation_layout(cfg)
    return D(observation_dim=dims, observation_names=names, output_mask_key="grippers", **kw)


def test_knn_in_place_is_opt_in():
    d = _data("rope")
    assert d.knn_in_place is False
    d.rebuild_every_call, d.consumer_accepts_capacity = True, True
    assert not d.refresh_in_place()  # the eager exact-size kNN rebuild stays the default


@pytest.mark.parametrize("task,precision,fused,hepi,flag",
                         list(itertools.product(("rope", "rigid"), ("fp32", "bf16"), (True, False), (True, False),
                                                (True, False))))
def test_refresh_in_place_truth_table(task, precision, fused, hepi, flag):
    """kNN edges are rebuilt in place with the flag, a HEPi policy, and either no num_valid (rope: exact set, any path)
    or the fused 16-bit edge path (rigid: fixed-capacity set); otherwise the eager rebuild stays."""
    from geometry_rl_b200 import ops
    d = _data(task)
    d.rebuild_every_call, d.knn_in_place, d.consumer_accepts_capacity = True, flag, hepi
    ops.set_precision(precision)
    ops.set_fused_edge(fused)
    try:
        want = flag and hepi and (task == "rope" or (precision == "bf16" and fused))
        assert d.refresh_in_place() == want
        d.rebuild_every_call = False
        assert not d.refresh_in_place()
        d.rebuild_every_call, d.build_edges = True, False
        assert not d.refresh_in_place()
    finally:
        ops.set_fused_edge(True)
        ops.set_precision("fp32")
