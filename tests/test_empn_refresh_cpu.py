"""CPU: the layout rules of the EMPN homogeneous views derived on the device (tests/homogeneous_reference.py) against the
long way round (oracle.graph's homogeneous_edge_index, masking and a stable sort as build_sub_edge_set does), and when
the data builders refresh them in place for EMPN."""
import itertools

import numpy as np
import pytest
import torch

from geometry_rl_b200.synthetic import CONFIGS, observation_layout
from tests.homogeneous_reference import edge_set_layouts, merge_layout, sub_layout, sub_long_way

SUB_FIELDS = ("eids", "eids32", "rowptr_dst", "edge_src", "edge_dst", "rowptr_src", "src_eid_parent", "edge_dst_parent",
              "s_src", "s_dst")


def _topology(B, P, A, num_points, seed):
    from oracle import graph as og
    gen = torch.Generator().manual_seed(seed)
    pv = {"object_geometry": torch.rand(B, P, 3, generator=gen), "grippers": torch.rand(B, A, 3, generator=gen),
          "target_geometry": torch.rand(B, P, 3, generator=gen)}
    return og.build_topology(og.TASKS["rigid"], pv, full_graph_obs=False, output_mask_key="grippers",
                             num_points=torch.as_tensor(num_points))


def _parts(g, capacity):
    """Per edge type: its COO as the data builder holds it - exact, or the in-place builder's fixed capacity (kNN
    INTERNAL B*P*k, TASK B*P*A) with zero tails."""
    offs, o = {}, 0
    for t in g.node_types:
        offs[t] = o
        o += g.nodes_per_graph[t]
    B, out = g.num_graphs, []
    for et in g.edge_types:
        src, kind, dst = et
        ei = g.edge_index_dict[et].numpy()
        cap = ei.shape[1]
        if capacity and kind != "agent":
            cap = B * g.nodes_per_graph[src] * (3 if kind == "internal" else g.nodes_per_graph[dst])
        coo = np.zeros((2, cap), np.int64)
        coo[:, :ei.shape[1]] = ei
        ptr = np.concatenate([[0], np.cumsum(g.edge_counts[et].numpy())]).astype(np.int64)
        out.append(dict(coo=coo, edge_ptr=ptr, n_src=g.nodes_per_graph[src], n_dst=g.nodes_per_graph[dst],
                        off_src=offs[src], off_dst=offs[dst]))
    return out


def _cases():
    P = 10
    return [("ragged_A1", 6, P, 1, [0, 1, P, 4, 2, 3]), ("ragged_A2", 6, P, 2, [P, 0, 1, 7, 3, 2]),
            ("all_empty_A1", 3, P, 1, [0, 0, 0]), ("all_empty_A2", 3, P, 2, [0, 1, 0]),
            ("full_A2", 2, P, 2, [P, P]), ("one_graph", 1, P, 1, [1])]


@pytest.mark.parametrize("case", range(6))
@pytest.mark.parametrize("capacity", [False, True])
def test_merge_rule_equals_the_oracle_homogeneous_view(case, capacity):
    name, B, P, A, nv = _cases()[case]
    g = _topology(B, P, A, nv, case)
    n_tot = P + A
    parts = _parts(g, capacity)
    cap = sum(p["coo"].shape[1] for p in parts)
    got = merge_layout(parts, B, n_tot, cap)
    ref = g.homogeneous_edge_index().numpy()
    E = ref.shape[1]
    counts = sum(g.edge_counts[et] for et in g.edge_types).numpy()
    assert np.array_equal(got["edge_ptr"], np.concatenate([[0], np.cumsum(counts)])), name
    assert got["coo"].shape == (2, cap) and (capacity or cap == E), name
    assert np.array_equal(got["coo"][:, :E], ref), name
    assert not got["coo"][:, E:].any(), name


@pytest.mark.parametrize("case", range(6))
@pytest.mark.parametrize("capacity", [False, True])
def test_sub_rule_equals_masking_and_a_stable_sort(case, capacity):
    name, B, P, A, nv = _cases()[case]
    g = _topology(B, P, A, nv, 10 + case)
    n_tot = P + A
    exact_parts = _parts(g, False)
    exact = merge_layout(exact_parts, B, n_tot, sum(p["coo"].shape[1] for p in exact_parts))
    parent_x = edge_set_layouts(exact["coo"], exact["edge_ptr"], B, n_tot)
    out_ids = (np.arange(B)[:, None] * n_tot + P + np.arange(A)).reshape(-1)
    ref = sub_long_way(parent_x, out_ids, B * n_tot)
    E_sub = ref["eids"].shape[0]
    if not capacity:
        got = sub_layout(parent_x, B, n_tot, P, A, E_sub)
        for f in SUB_FIELDS:
            assert got[f].shape == ref[f].shape and np.array_equal(got[f], ref[f]), (name, f)
        return
    parts = _parts(g, True)
    cap_parent = sum(p["coo"].shape[1] for p in parts)
    merged = merge_layout(parts, B, n_tot, cap_parent)
    parent = edge_set_layouts(merged["coo"], merged["edge_ptr"], B, n_tot)
    E = int(exact["edge_ptr"][B])
    for f in ("rowptr_dst", "rowptr_src"):  # the capacity parent equals the exact one over its real edges
        assert np.array_equal(parent[f], parent_x[f]), (name, f)
    for f in ("edge_src", "edge_dst", "eid_coo", "src_eid", "s_src", "s_dst"):
        assert np.array_equal(parent[f][:E], parent_x[f]), (name, f)
    cap = sum(p["coo"].shape[1] for p, (_, _, dst) in zip(parts, g.edge_types) if dst == "grippers")
    assert cap >= E_sub
    got = sub_layout(parent, B, n_tot, P, A, cap)
    for f in ("rowptr_dst", "rowptr_src"):
        assert np.array_equal(got[f], ref[f]), (name, f)
    assert np.array_equal(got["edge_dst_parent"][:E], ref["edge_dst_parent"]), name
    assert (got["edge_dst_parent"][E:] == -1).all(), name
    for f in SUB_FIELDS:
        if f not in ("rowptr_dst", "rowptr_src", "edge_dst_parent"):
            assert np.array_equal(got[f][:E_sub], ref[f]), (name, f)
    # tails: 0 where the parent holds 0, else what a gather through those zeros reads
    for f in ("eids", "eids32", "edge_src"):
        assert not got[f][E_sub:].any(), (name, f)
    assert (got["edge_dst"][E_sub:] == got["edge_dst_parent"][0]).all(), name
    assert (got["src_eid_parent"][E_sub:] == got["eids32"][0]).all(), name
    assert (got["s_src"][E_sub:] == got["edge_src"][0]).all() and (got["s_dst"][E_sub:] == got["edge_dst"][0]).all()


def _data(task, **kw):
    if task == "rope":
        from geometry_rl_b200.modules.pyg_data.rope_tasks_data import RopeTasksData as D
        cfg = CONFIGS["rope_shaping_hepi_trpl_cfg"]
    else:
        from geometry_rl_b200.modules.pyg_data.rigid_tasks_data import RigidTasksData as D
        cfg = CONFIGS["rigid_pushing_multi_empn_trpl_cfg"]
    dims, names = observation_layout(cfg)
    return D(observation_dim=dims, observation_names=names, output_mask_key="grippers", **kw)


def test_empn_policy_wrapper_accepts_the_capacity_homogeneous_view():
    from geometry_rl_b200 import learner
    actor, *_ = learner.build_agent(CONFIGS["rigid_pushing_multi_empn_trpl_cfg"], torch.device("cpu"), seed=0)
    hd = actor.get_submodule("0").module.hyper_data
    assert hd.consumer_accepts_homogeneous_capacity and not hd.consumer_accepts_capacity
    actor, *_ = learner.build_agent(CONFIGS["rigid_insertion_multi_hepi_trpl_cfg"], torch.device("cpu"), seed=0)
    assert not actor.get_submodule("0").module.hyper_data.consumer_accepts_homogeneous_capacity


@pytest.mark.parametrize("task,precision,fused,flag,internal",
                         list(itertools.product(("rope", "rigid"), ("fp32", "bf16"), (True, False), (True, False),
                                                ("knn", "radius"))))
def test_refresh_in_place_truth_table_for_the_homogeneous_consumer(task, precision, fused, flag, internal):
    """EMPN: kNN INTERNAL edges with the flag on the fused 16-bit edge path are rebuilt in place; radius edges, the
    strict fp32 or unfused path, or no flag keep the eager rebuild."""
    from geometry_rl_b200 import ops
    d = _data(task, internal_edges=internal, radius=0.1 if internal == "radius" else None)
    d.rebuild_every_call, d.knn_in_place, d.consumer_accepts_homogeneous_capacity = True, flag, True
    ops.set_precision(precision)
    ops.set_fused_edge(fused)
    try:
        want = flag and internal == "knn" and precision == "bf16" and fused
        assert d.refresh_in_place() == want
        d.rebuild_every_call = False
        assert not d.refresh_in_place()
        d.rebuild_every_call, d.build_edges = True, False
        assert not d.refresh_in_place()
        d.build_edges, d.consumer_accepts_homogeneous_capacity = True, False
        assert not d.refresh_in_place()  # neither consumer: the eager rebuild
    finally:
        ops.set_fused_edge(True)
        ops.set_precision("fp32")


def test_homo_part_layout_matches_the_c_compiler():
    import ctypes as C
    import os
    import subprocess
    import tempfile
    from geometry_rl_b200 import _lib as L
    header = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "grl_b200.h")
    lines = ["#include <stdio.h>", "#include <stddef.h>", f'#include "{header}"', "int main(void) {",
             'printf("size %zu\\n", sizeof(GrlHomoPart));',
             'printf("max %d\\n", GRL_MAX_HOMO_PARTS);']
    lines += [f'printf("{f} %zu\\n", offsetof(GrlHomoPart, {f}));' for f, _ in L.GrlHomoPart._fields_]
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "t.c"), os.path.join(d, "t")
        open(src, "w").write("\n".join(lines + ["return 0; }"]))
        subprocess.run(["gcc", src, "-o", exe], check=True)
        out = dict(l.split() for l in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(out["size"]) == C.sizeof(L.GrlHomoPart) and int(out["max"]) == L.HOMO_MAX_PARTS
    for f, _ in L.GrlHomoPart._fields_:
        assert int(out[f]) == getattr(L.GrlHomoPart, f).offset, f
