"""CPU: the radius-graph brute force (tests/radius_oracle.py) and the data builders' radius / rebuild arguments."""
import math

import pytest
import torch

from geometry_rl_b200.synthetic import CONFIGS, observation_layout


def _rope_data(**kw):
    from geometry_rl_b200.modules.pyg_data.rope_tasks_data import RopeTasksData
    dims, names = observation_layout(CONFIGS["rope_shaping_hepi_trpl_cfg"])
    return RopeTasksData(observation_dim=dims, observation_names=names, output_mask_key="grippers", **kw)


def test_oracle_radius_edges():
    from tests.radius_oracle import radius_edges
    # points on a line at 0, 0.5, 1.0, 1.5 (exact fp32 distances): radius 0.5 includes the neighbours at exactly 0.5
    pts = torch.tensor([[0.0, 0, 0], [0.5, 0, 0], [1.0, 0, 0], [1.5, 0, 0]])
    ei = radius_edges(pts, 0.5, 8)
    assert ei.tolist() == [[0, 1, 1, 2, 2, 3], [1, 0, 2, 1, 3, 2]]  # (source j, target i), sorted by (j, i)
    # saturation with a tie: centre 1 has 0 and 2 at the same distance, max 1 neighbour -> the lower index (0)
    ei = radius_edges(pts, 0.5, 1)
    assert [tuple(e) for e in ei.t().tolist() if e[1] == 1] == [(0, 1)]
    # a NaN point has no edges, and no point has it as a neighbour
    nan = pts.clone()
    nan[2, 1] = float("nan")
    ei = radius_edges(nan, 0.5, 8)
    assert ei.tolist() == [[0, 1], [1, 0]]
    assert radius_edges(pts[:1], 1.0, 8).shape == (2, 0) and radius_edges(pts[:0], 1.0, 8).shape == (2, 0)


def test_oracle_build_topology_radius_option():
    from oracle import graph as og
    from tests.radius_oracle import radius_edges, radius_topology
    B, P, A = 2, 4, 2
    line = torch.tensor([[0.0, 0, 0], [0.5, 0, 0], [1.0, 0, 0], [5.0, 0, 0]])
    pv = {"links": line.expand(B, -1, -1), "grippers": torch.zeros(B, A, 3), "target_geometry": torch.zeros(B, P, 3)}
    g = radius_topology(og.ROPE, pv, full_graph_obs=False, output_mask_key="grippers", radius=0.5, max_num_neighbors=8)
    et = ("links", "internal", "links")
    assert g.edge_counts[et].tolist() == [4, 4]  # 0-1, 1-2 both ways; the point at 5.0 is isolated
    assert torch.equal(g.edge_index_dict[et][:, 4:], radius_edges(line, 0.5, 8) + P)
    knn = og.build_topology(og.ROPE, pv, full_graph_obs=False, output_mask_key="grippers")
    assert knn.edge_counts[et].tolist() == [12, 12]


def test_defaults_keep_knn_and_build_once():
    d = _rope_data()
    assert d.internal_edges == "knn" and d.radius is None and not d.rebuild_every_call
    assert not d.refresh_in_place()


@pytest.mark.parametrize("kw,match", [
    (dict(internal_edges="ball"), "internal_edges"),
    (dict(internal_edges="radius"), "radius > 0"),
    (dict(internal_edges="radius", radius=0.0), "radius > 0"),
    (dict(internal_edges="radius", radius=-1.0), "radius > 0"),
    (dict(internal_edges="radius", radius=math.nan), "radius > 0"),
    (dict(internal_edges="radius", radius=math.inf), "radius > 0"),
    (dict(internal_edges="radius", radius=True), "radius > 0"),
    (dict(internal_edges="radius", radius=0.1, max_num_neighbors=0), "max_num_neighbors"),
    (dict(internal_edges="radius", radius=0.1, max_num_neighbors=9), "max_num_neighbors"),
    (dict(internal_edges="radius", radius=0.1, max_num_neighbors=4.0), "max_num_neighbors"),
    (dict(radius=0.1), "only used with internal_edges='radius'"),
])
def test_radius_arguments_are_validated_at_construction(kw, match):
    with pytest.raises(ValueError, match=match):
        _rope_data(**kw)


def test_cloth_internal_edges_stay_full():
    from geometry_rl_b200.modules.pyg_data.cloth_tasks_data import ClothTasksData
    dims, names = observation_layout(CONFIGS["cloth_hanging_multi_hepi_trpl_cfg"])
    with pytest.raises(ValueError, match="full"):
        ClothTasksData(observation_dim=dims, observation_names=names, internal_edges="radius", radius=0.1)


def test_refresh_in_place_only_on_the_fused_16bit_path_with_radius_edges():
    from geometry_rl_b200 import ops
    d = _rope_data(internal_edges="radius", radius=0.025, max_num_neighbors=8)
    d.rebuild_every_call = True
    ops.set_precision("bf16")
    try:
        assert not d.refresh_in_place()  # no model that consumes fixed-capacity edge sets attached
        d.consumer_accepts_capacity = True
        assert d.refresh_in_place() == ops.fused_edge_enabled()
        ops.set_fused_edge(False)
        assert not d.refresh_in_place()  # materialised-basis pair: exact topology
        ops.set_fused_edge(True)
        d.rebuild_every_call = False
        assert not d.refresh_in_place()
    finally:
        ops.set_fused_edge(True)
        ops.set_precision("fp32")
    d.rebuild_every_call = True
    assert not d.refresh_in_place()  # strict fp32 path: exact topology
    k = _rope_data()
    k.rebuild_every_call, k.consumer_accepts_capacity = True, True
    assert not k.refresh_in_place()  # kNN: eager rebuild


def test_hepi_policy_wrapper_accepts_capacity_edge_sets():
    from geometry_rl_b200 import learner
    cfg = CONFIGS["rope_shaping_hepi_trpl_cfg"]
    actor, *_ = learner.build_agent(cfg, torch.device("cpu"))
    assert actor.get_submodule("0").module.hyper_data.consumer_accepts_capacity
    cfg = CONFIGS["rigid_pushing_multi_empn_trpl_cfg"]
    actor, *_ = learner.build_agent(cfg, torch.device("cpu"))
    assert not actor.get_submodule("0").module.hyper_data.consumer_accepts_capacity  # EMPN: homogeneous view, exact
