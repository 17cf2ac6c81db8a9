"""GPU: the EMPN homogeneous views derived on the device (ops.homogeneous_edge_set / ops.sub_edge_set) and rebuilt in
place with the kNN topology (`rebuild_every_call` + `knn_in_place`), inside the captured update and the acting graph.

Integer topology is compared with torch.equal against today's torch-op views (GraphBatch.homogeneous() and
build_sub_edge_set on an exact batch); output buffers are pre-filled with a sentinel first, so an entry the kernels do
not write shows.  16-bit steps are held to north_star's bound against the oracle, as in test_gpu_knn_refresh.py."""
import dataclasses

import numpy as np
import pytest
import torch

from geometry_rl_b200.synthetic import CONFIGS
from tests import gpu_helpers as G
from tests.homogeneous_reference import edge_set_layouts, merge_layout, sub_layout
from tests.test_gpu_knn_refresh import _agent, _num_valid, _positions, _run

pytestmark = pytest.mark.gpu

EMPN = "rigid_pushing_multi_empn_trpl_cfg"
OBJ, GRIP = "object_geometry", "grippers"
ET = ((OBJ, "internal", OBJ), (GRIP, "agent", GRIP), (OBJ, "task", GRIP))
FIELDS = ("coo", "edge_ptr", "rowptr_dst", "edge_src", "edge_dst", "eid_coo", "rowptr_src", "src_eid", "s_src", "s_dst")
SUB_FIELDS = ("out_ids", "eids", "eids32", "rowptr_dst", "edge_src", "edge_dst", "rowptr_src", "src_eid_parent",
              "edge_dst_parent", "s_src", "s_dst")
SENTINEL = 0x5A5A5A5A


@pytest.fixture
def sixteen_bit():
    from geometry_rl_b200 import ops
    ops.set_precision("bf16")
    yield
    ops.set_precision("fp32")


def _graph(pts, nv, A, in_place):
    """The rigid topology as RigidTasksData builds it: exact (build once / eager rebuild) or the in-place builder's sets
    (fixed-capacity kNN INTERNAL and TASK edges, marked refreshed)."""
    from geometry_rl_b200 import ops
    from geometry_rl_b200.modules.pyg_data.graph import GraphBatch
    B, P, _ = pts.shape
    dev = pts.device
    g = GraphBatch(B, {OBJ: P, GRIP: A}, dev)
    if in_place:
        g.add_edge_set(ET[0], ops.knn_edge_set(pts, nv, 3), refreshed=True)
    else:
        g.add_edge_type(ET[0], *ops.knn_graph(pts, nv, 3))
    if A > 1:
        g.add_edge_type(ET[1], *ops.dense_edges(0, B, A, A, dev))
    else:
        g.add_edge_type(ET[1], torch.empty(2, 0, dtype=torch.int64, device=dev),
                        torch.zeros(B + 1, dtype=torch.int64, device=dev))
    coo, ptr = ops.dense_edges(1, B, P, A, dev, num_valid=nv, capacity=in_place)
    g.add_edge_type(ET[2], coo, ptr, refreshed=in_place, exact=not in_place)
    g.output_mask_key, g.output_mask = GRIP, slice(P, P + A)
    return g


def _refresh(g, pts, nv):
    from geometry_rl_b200 import ops
    B, P, _ = pts.shape
    ops.refresh_knn_edge_set(g.edge_sets[ET[0]], pts, nv, 3)
    ops.refresh_edge_set(g.edge_sets[ET[2]], *ops.dense_edges(1, B, P, g.nodes_per_graph[GRIP], pts.device,
                                                              num_valid=nv, capacity=True))
    g.refresh_homogeneous()


def _poison(obj, fields):
    for f in fields:
        t = getattr(obj, f)
        if t is not None and t.numel():
            t.fill_(SENTINEL)


def _inputs(B, A):
    P = 48
    return _positions(B, P, 100 + B + A), _num_valid(B, P, 200 + B + A), A


def _check_capacity_set(es, ref, what):
    """`es` (fixed capacity) against the exact `ref` of the same batch: full CSR row pointers, real prefixes, tails."""
    from geometry_rl_b200 import ops
    ops.src_sorted_pairs(ref)
    E = ref.n_edges
    assert not es.exact and es.n_edges >= E and (es.n_src, es.n_dst) == (ref.n_src, ref.n_dst), what
    for f in ("edge_ptr", "rowptr_dst", "rowptr_src"):
        assert torch.equal(getattr(es, f), getattr(ref, f)), (what, f)
    assert torch.equal(es.coo[:, :E], ref.coo), what
    for f in ("edge_src", "edge_dst", "eid_coo", "src_eid", "s_src", "s_dst"):
        assert torch.equal(getattr(es, f)[:E], getattr(ref, f)), (what, f)
    assert not bool(es.coo[:, E:].any()), what
    for f in ("edge_src", "eid_coo", "src_eid"):
        assert not bool(getattr(es, f)[E:].any()), (what, f)
    assert bool((es.edge_dst[E:] == es.coo[1, 0]).all()), what
    assert bool((es.s_src[E:] == es.edge_src[0]).all()) and bool((es.s_dst[E:] == es.edge_dst[0]).all()), what


@pytest.mark.parametrize("A", [1, 2])
@pytest.mark.parametrize("B", [1, 37, 4096])
def test_merge_equals_homogeneous(B, A):
    from geometry_rl_b200 import ops
    pts, nv, A = _inputs(B, A)
    P = pts.shape[1]
    exact = _graph(pts, nv, A, False)
    ref = exact.homogeneous()
    ops.src_sorted_pairs(ref)
    # exact inputs: the device merge equals the torch-op view array for array
    es = ops.homogeneous_edge_set(exact._homo_parts(), B, P + A)
    _poison(es, FIELDS)
    ops.refresh_homogeneous_edge_set(es, exact._homo_parts())
    assert es.exact and (es.n_src, es.n_dst, es.n_edges) == (ref.n_src, ref.n_dst, ref.n_edges)
    for f in FIELDS:
        assert torch.equal(getattr(es, f), getattr(ref, f)), f
    # the in-place builder's capacity sets of the same batch
    g = _graph(pts, nv, A, True)
    es = g.homogeneous()
    assert es.n_edges == sum(s.n_edges for s in g.edge_sets.values())
    _poison(es, FIELDS)
    g.refresh_homogeneous()
    _check_capacity_set(es, ref, "capacity")
    if B <= 37:  # the numpy restatement of the rules, tails included
        parts = [dict(coo=s.coo.cpu().numpy(), edge_ptr=s.edge_ptr.cpu().numpy(), n_src=s.n_src // B, n_dst=s.n_dst // B,
                      off_src=o_s, off_dst=o_d) for s, o_s, o_d in g._homo_parts()]
        m = merge_layout(parts, B, P + A, es.n_edges)
        want = edge_set_layouts(m["coo"], m["edge_ptr"], B, P + A)
        for f in FIELDS:
            assert np.array_equal(getattr(es, f).cpu().numpy(), want[f]), f


@pytest.mark.parametrize("A", [1, 2])
@pytest.mark.parametrize("B", [1, 37, 4096])
def test_sub_set_equals_build_sub_edge_set(B, A):
    from geometry_rl_b200 import ops
    pts, nv, A = _inputs(B, A)
    P = pts.shape[1]
    H = _graph(pts, nv, A, False).homogeneous()
    out_ids = (torch.arange(B, device="cuda")[:, None] * (P + A) + P + torch.arange(A, device="cuda")).reshape(-1)
    ref = ops.build_sub_edge_set(H, out_ids)
    ops.src_sorted_pairs(H, ref)
    sub = ops.sub_edge_set(H, P, A, ref.n_edges)
    _poison(sub, SUB_FIELDS[1:] + ("edge_ptr",))
    ops.refresh_sub_edge_set(sub, H, P)
    assert sub.exact and (sub.n_src, sub.n_dst, sub.n_edges) == (ref.n_src, ref.n_dst, ref.n_edges)
    for f in SUB_FIELDS:
        assert torch.equal(getattr(sub, f), getattr(ref, f)), f
    # from the in-place builder's capacity parent: every row kept, the same sub set over the real edges
    g = _graph(pts, nv, A, True)
    pr = g.homogeneous_pruned()
    sub, es = pr.sub, pr.es
    assert pr.live_ids is None and pr.live_ids32 is None and es is g.homogeneous() and not sub.exact
    _poison(sub, SUB_FIELDS[1:] + ("edge_ptr",))
    g.refresh_homogeneous()
    E, E_par = ref.n_edges, H.n_edges
    assert torch.equal(sub.out_ids, ref.out_ids)
    for f in ("rowptr_dst", "rowptr_src"):
        assert torch.equal(getattr(sub, f), getattr(ref, f)), f
    for f in ("eids", "eids32", "edge_src", "edge_dst", "src_eid_parent", "s_src", "s_dst"):
        assert torch.equal(getattr(sub, f)[:E], getattr(ref, f)), f
    assert torch.equal(sub.edge_dst_parent[:E_par], ref.edge_dst_parent)
    assert bool((sub.edge_dst_parent[E_par:] == -1).all())
    for f in ("eids", "eids32", "edge_src"):
        assert not bool(getattr(sub, f)[E:].any()), f
    assert bool((sub.edge_dst[E:] == sub.edge_dst_parent[0]).all())
    assert bool((sub.src_eid_parent[E:] == sub.eids32[0]).all())
    assert bool((sub.s_src[E:] == sub.edge_src[0]).all()) and bool((sub.s_dst[E:] == sub.edge_dst[0]).all())
    if B <= 37:
        parent = {f: getattr(es, f).cpu().numpy() for f in ("rowptr_dst", "edge_src", "edge_dst")}
        want = sub_layout(parent, B, P + A, P, A, sub.n_edges)
        for f in SUB_FIELDS[1:]:
            assert np.array_equal(getattr(sub, f).cpu().numpy(), want[f]), f


def test_captured_refresh_follows_new_positions_and_num_valid():
    B, P, A = 96, 48, 2
    pts, nv = _positions(B, P, 31), _num_valid(B, P, 32)
    g = _graph(pts, nv, A, True)
    pr = g.homogeneous_pruned()
    es, sub = pr.es, pr.sub
    ptrs = {f: getattr(es, f).data_ptr() for f in FIELDS}
    ptrs.update({"sub." + f: getattr(sub, f).data_ptr() for f in SUB_FIELDS + ("edge_ptr",)})
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        _refresh(g, pts, nv)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _refresh(g, pts, nv)
    for seed in (33, 34):
        pts.copy_(_positions(B, P, seed))
        nv.copy_(_num_valid(B, P, seed + 10))
        graph.replay()
        torch.cuda.synchronize()
        now = {f: getattr(es, f).data_ptr() for f in FIELDS}
        now.update({"sub." + f: getattr(sub, f).data_ptr() for f in SUB_FIELDS + ("edge_ptr",)})
        assert now == ptrs
        fresh = _graph(pts, nv, A, True).homogeneous_pruned()
        for f in FIELDS:
            assert torch.equal(getattr(es, f), getattr(fresh.es, f)), (seed, f)
        for f in SUB_FIELDS + ("edge_ptr",):
            assert torch.equal(getattr(sub, f), getattr(fresh.sub, f)), (seed, f)
        _check_capacity_set(es, _graph(pts, nv, A, False).homogeneous(), f"replay {seed}")


def _empn_data(cfg, in_place):
    data = G.make_data(cfg, policy=True)
    if in_place:
        data.consumer_accepts_homogeneous_capacity, data.rebuild_every_call, data.knn_in_place = True, True, True
        assert data.refresh_in_place()
    return data


def test_body_in_place_equals_exact_pruned_evaluation(sixteen_bit):
    """EMPN outputs and every parameter gradient with the in-place views (every row kept, last layer through the refreshed
    sub set) against the exact pruned evaluation on the same batch, at test_pruned_rows_equal_dense_evaluation's bf16
    bound; the one-time calibration gives bit-identical parameters."""
    from geometry_rl_b200.synthetic import synthetic_obs
    cfg, B = CONFIGS[EMPN], 72
    gen = torch.Generator().manual_seed(21)
    obs = synthetic_obs(cfg, B, gen, env_ids=torch.arange(B) * max(1, cfg.num_envs // B))
    torch.manual_seed(5)
    net = G.make_policy_body(cfg)
    init = {k: v.clone() for k, v in net.state_dict().items()}
    calibrated = {}
    for in_place in (False, True):  # the calibration forward (train mode) from the same initial parameters
        net.load_state_dict(init)
        net.train()
        graph, u = _empn_data(cfg, in_place).build_data(*G.obs_args(cfg, obs, policy=True), train=False)
        with torch.no_grad():
            net.one_step(graph, u)
        calibrated[in_place] = {k: v.clone() for k, v in net.state_dict().items()}
    for k in calibrated[False]:
        assert torch.equal(calibrated[True][k], calibrated[False][k]), k
    with torch.no_grad():
        for n, p in net.named_parameters():
            if n.endswith("bias") and float(p.abs().max()) == 0:
                p.normal_(0, 0.05)
    net.eval()
    res = {}
    for in_place in (False, True):
        data = _empn_data(cfg, in_place)
        args = G.obs_args(cfg, obs, policy=True)
        if in_place:  # a first batch builds the views, the batch compared is a refresh
            data.build_data(*G.obs_args(cfg, synthetic_obs(cfg, B, torch.Generator().manual_seed(3)), policy=True),
                            train=False)
        graph, u = data.build_data(*args, train=False)
        pr = graph.homogeneous_pruned()
        assert (pr.live_ids is None) == in_place
        net.zero_grad(set_to_none=True)
        out, hidden = net.one_step(graph, u)
        if not in_place:
            w_out = torch.randn(out.shape, generator=gen).cuda()
            w_hid = torch.randn(hidden.shape, generator=gen).cuda()
        ((out * w_out).sum() + (hidden * w_hid).sum()).backward()
        res[in_place] = (out.detach().clone(), hidden.detach().clone(),
                         {k: p.grad.detach().clone() for k, p in net.named_parameters() if p.grad is not None})
    (o0, h0, g0), (o1, h1, g1) = res[False], res[True]
    tol = 4e-3
    assert G.rel(o1, o0) < tol, G.err_report("out", o1, o0)
    assert G.rel(h1, h0) < tol, G.err_report("hidden", h1, h0)
    assert set(g0) == set(g1)
    bad = [G.err_report(k, g1[k], g0[k]) for k in g0 if G.rel(g1[k], g0[k]) >= tol]
    assert not bad, "\n".join(bad)


def test_captured_16bit_update_matches_oracle_and_eager(sixteen_bit):
    from tests.test_gpu_step16 import _compare
    graphed, eager = _run(EMPN, 24, "graphed"), _run(EMPN, 24, "eager_in_place")
    for (lg, fg, _, (out, ref)), (le, fe, _, _) in zip(graphed, eager):
        pol = {k[len("actor.0.module."):]: v for k, v in fg.items() if k.startswith("actor.0.module.")}
        vf = {k[len("critic.module._network1."):]: v for k, v in fg.items() if k.startswith("critic.module._network1.")}
        report = []
        bad = _compare(out, ref[0], pol, ref[1], vf, ref[2], report)
        assert not bad, "\n".join(bad + ["--"] + report)
        assert lg == le  # the same in-place rebuild replayed or launched eagerly
        for k in fe:
            assert torch.equal(fg[k], fe[k]), k


def test_fit_over_minibatches_with_different_num_valid(sixteen_bit):
    """Learner.fit replaying the captured update over a buffer whose minibatches hold different point counts equals the
    same epochs through the eager `update` with the same in-place rebuild, bit for bit."""
    from geometry_rl_b200 import learner
    from geometry_rl_b200.rollout import DeviceRolloutBuffer
    from geometry_rl_b200.tensors import to_device
    from oracle.step import OracleAgent, make_minibatch
    n_frames, mb_size = 96, 32
    finals = []
    for graphed in (True, False):
        torch.manual_seed(0)
        cfg, actor, critic, loss_module, obs, gen, hd = _agent(EMPN, n_frames, seed=6)
        assert hd.refresh_in_place()
        frames = to_device(make_minibatch(cfg, OracleAgent(cfg, actor.state_dict(), critic.state_dict()), obs, gen),
                           G.dev())
        frames = {k: v for k, v in frames.items() if torch.is_tensor(v)}
        nv = obs["infos"][:, 0]
        assert len(set(nv.tolist())) > 1
        buf = DeviceRolloutBuffer(n_frames, mb_size, G.dev(), drop_last=True, generator=torch.Generator().manual_seed(7))
        buf.extend(frames)
        lrn = learner.Learner(dataclasses.replace(cfg, clip_grad_norm=False), actor, critic, loss_module,
                              overlap_critic=False)
        res = lrn.fit(buf, epochs=2, graphed=graphed)
        assert len(res) == 2 * (n_frames // mb_size)
        torch.cuda.synchronize()
        finals.append(torch.cat([p.detach().reshape(-1).clone() for p in list(actor.parameters()) + list(critic.parameters())]))
    assert bool(torch.isfinite(finals[0]).all())
    assert torch.equal(finals[0], finals[1])


def test_act_graph_with_in_place_views(sixteen_bit):
    """capture_act + act_graphed == eager act at the same Philox state, act replays interleaved with update replays; and
    within the 16-bit bound of eager act on the eager exact topology."""
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    from oracle.step import OracleAgent, make_minibatch
    from tests.test_gpu_act import _obs_batches, _outs
    cfg, actor, critic, loss_module, obs, gen, hd = _agent(EMPN, 6, seed=4)
    assert hd.refresh_in_place()
    _, exact_actor, _, _, _, _, exact_hd = _agent(EMPN, 6, seed=4, in_place=False)
    exact_actor.load_state_dict(actor.state_dict())
    assert not exact_hd.refresh_in_place()
    batches = _obs_batches(cfg, 6, 4, 900)
    actor.capture_act(batches[0], seed=31)
    lrn = learner.Learner(cfg, actor, critic, loss_module)
    mb = to_device(make_minibatch(cfg, OracleAgent(cfg, actor.state_dict(), critic.state_dict()), obs, gen), G.dev())
    lrn.capture(mb, warmup=2)
    graphed = []
    for i, td in enumerate(batches[1:]):
        state = actor.act_state()
        replayed, eager, exact = dict(td), dict(td), dict(td)
        actor.act_graphed(replayed)
        actor.set_act_state(*state)
        actor.act(eager)
        for got, exp in zip(_outs(replayed), _outs(eager)):
            assert torch.equal(got, exp), i
        exact_actor.load_state_dict(actor.state_dict())
        exact_actor.set_act_state(*state)
        exact_actor.act(exact)
        for name, got, exp in zip(("loc", "cov", "action", "log_prob"), _outs(replayed), _outs(exact)):
            assert G.rel(got, exp) < 1e-2, G.err_report(name, got, exp)
        graphed.append(_outs(replayed))
        lrn.update_graphed(mb)  # the update graph rewrites the shared placeholder from its own positions
    assert not torch.equal(graphed[0][0], graphed[1][0])


def test_capture_guard_keeps_radius_edges_eager(sixteen_bit):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    from tests.test_gpu_act import _obs_batches
    cfg = CONFIGS[EMPN]
    actor, critic, _, loss_module, _ = learner.build_agent(cfg, G.dev(), seed=0)
    hd = actor.get_submodule("0").module.hyper_data
    hd.rebuild_every_call, hd.knn_in_place, hd.internal_edges, hd.radius = True, True, "radius", 0.05
    assert not hd.refresh_in_place()
    obs = _obs_batches(cfg, 4, 1, 5)[0]
    lrn = learner.Learner(cfg, actor, critic, loss_module)
    with pytest.raises(ValueError, match="cannot be replayed"):
        lrn.capture({k: v for k, v in to_device(obs, G.dev()).items()})
    with pytest.raises(ValueError, match="cannot be replayed"):
        actor.capture_act(obs, seed=0)
