"""GPU: radius-graph topology (ops.radius_graph, `internal_edges="radius"`) and its in-place refresh on every call
(`rebuild_every_call` on the fused 16-bit path), captured in the CUDA graph of the update.

Integer topology is compared bit-exactly with the CPU brute force (tests/radius_oracle.py); update steps on a radius
topology within north_star's 16-bit bound (1e-2 of each tensor's max magnitude), as in test_gpu_step16.py."""
import pytest
import torch

from geometry_rl_b200.synthetic import CONFIGS, synthetic_obs
from tests import gpu_helpers as G

pytestmark = pytest.mark.gpu

ROPE, RIGID = "rope_shaping_hepi_trpl_cfg", "rigid_insertion_multi_hepi_trpl_cfg"
# rope links are ~0.010 apart (degree ~4 at 0.025); rigid object points ~0.04 (valid points only)
RADIUS = {ROPE: (0.025, 8), RIGID: (0.08, 6)}


@pytest.fixture
def sixteen_bit():
    from geometry_rl_b200 import ops
    ops.set_precision("bf16")
    yield
    ops.set_precision("fp32")


def _oracle_radius(pos, nv, r, m):
    from tests.radius_oracle import radius_edges
    B, P, _ = pos.shape
    parts = [radius_edges(pos[b, : int(nv[b]) if nv is not None else P], r, m) + b * P for b in range(B)]
    counts = torch.tensor([p.shape[1] for p in parts], dtype=torch.int64)
    return torch.cat(parts, dim=1), torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(counts, 0)])


def _cases():
    gen = torch.Generator().manual_seed(3)
    P = 27
    out = []
    # ragged num_valid: 0, 1, 2, a few, full
    pos = torch.randn(6, P, 3, generator=gen) * 0.5
    out.append(("ragged", pos, torch.tensor([0, 1, 2, 5, 27, 13], dtype=torch.int32), 0.6, 4))
    # a lattice with spacing 0.5 (exact fp32 distances): neighbours exactly at the radius are in (<=), and with
    # max_num_neighbors 2 the six lattice neighbours at equal distance saturate -> ties go to the lower index
    g = torch.stack(torch.meshgrid(torch.arange(3.), torch.arange(3.), torch.arange(3.), indexing="ij"), -1).reshape(-1, 3)
    lat = (g * 0.5).expand(2, -1, -1).contiguous()
    out.append(("lattice_at_radius", lat, None, 0.5, 8))
    out.append(("lattice_saturated", lat, None, 0.5, 2))
    # isolated points (far apart) and a NaN point (no edges, no error)
    iso = torch.randn(3, P, 3, generator=gen) * 0.3
    iso[0, 4] = torch.tensor([50.0, 50.0, 50.0])
    iso[1, 7, 1] = float("nan")
    iso[2] *= 100.0
    out.append(("isolated_nan", iso, torch.tensor([27, 27, 20], dtype=torch.int32), 0.35, 8))
    return out


@pytest.mark.parametrize("case", range(4))
def test_radius_graph_matches_oracle(case):
    from geometry_rl_b200 import ops
    name, pos, nv, r, m = _cases()[case]
    exp_coo, exp_ptr = _oracle_radius(pos, nv, r, m)
    nv_d = nv.cuda() if nv is not None else None
    coo, ptr = ops.radius_graph(pos.cuda(), nv_d, r, m)
    assert torch.equal(ptr.cpu(), exp_ptr), name
    assert torch.equal(coo.cpu(), exp_coo), name
    # the same neighbour sets as radius_neighbors
    nbr, cnt = ops.radius_neighbors(pos.cuda(), nv_d, r, m)
    B, P, _ = pos.shape
    pairs = {(b * P + int(j), b * P + i) for b in range(B) for i in range(P)
             for j in nbr[b, i, : int(cnt[b, i])].cpu().tolist()}
    assert pairs == set(map(tuple, coo.cpu().t().tolist())), name
    if name == "isolated_nan":
        assert not bool((coo.cpu() == 1 * P + 7).any()), "a NaN point has no edges"
    if name == "lattice_at_radius":
        assert int(cnt[0, 13]) == 6  # centre of the 3x3x3 lattice: six neighbours exactly at the radius


def test_capacity_mode_zero_tails_and_exact_prefix():
    from geometry_rl_b200 import ops
    name, pos, nv, r, m = _cases()[0]
    B, P, _ = pos.shape
    coo_x, ptr_x = ops.radius_graph(pos.cuda(), nv.cuda(), r, m)
    coo_c, ptr_c = ops.radius_graph(pos.cuda(), nv.cuda(), r, m, capacity=B * P * m)
    E = coo_x.shape[1]
    assert coo_c.shape == (2, B * P * m) and torch.equal(ptr_c, ptr_x)
    assert torch.equal(coo_c[:, :E], coo_x) and not bool(coo_c[:, E:].any())
    ex = ops.build_edge_set(coo_x, ptr_x, B, P, P)
    ca = ops.build_edge_set(coo_c, ptr_c, B, P, P, exact=False)
    assert ca.n_edges == B * P * m and not ca.exact and int(ca.rowptr_dst[-1]) == E
    for f in ("rowptr_dst", "rowptr_src"):
        assert torch.equal(getattr(ca, f), getattr(ex, f)), f
    for f in ("edge_src", "edge_dst", "eid_coo", "src_eid"):
        assert torch.equal(getattr(ca, f)[:E], getattr(ex, f)), f
    for f in ("edge_src", "eid_coo", "src_eid"):
        assert not bool(getattr(ca, f)[E:].any()), f + " tail"
    assert bool((ca.edge_dst[E:] >= 0).all() and (ca.edge_dst[E:] < ca.n_dst).all())  # gathered through a 0: in bounds
    # a smaller capacity drops the edges that do not fit and stays in bounds
    coo_s, ptr_s = ops.radius_graph(pos.cuda(), nv.cuda(), r, m, capacity=E // 2)
    assert int(ptr_s[-1]) == E // 2 and torch.equal(coo_s, coo_x[:, : E // 2])
    # in-place refresh from another point set: same tensors, contents of a fresh build
    pos2 = pos + 0.05 * torch.randn(pos.shape, generator=torch.Generator().manual_seed(9))
    ptrs = {f: getattr(ca, f).data_ptr() for f in ("coo", "rowptr_dst", "edge_src", "edge_dst", "src_eid")}
    ops.src_sorted_pairs(ca)
    coo2, ptr2 = ops.radius_graph(pos2.cuda(), nv.cuda(), r, m, capacity=B * P * m)
    ops.refresh_edge_set(ca, coo2, ptr2)
    fresh = ops.build_edge_set(*ops.radius_graph(pos2.cuda(), nv.cuda(), r, m), B, P, P)
    E2 = fresh.n_edges
    assert {f: getattr(ca, f).data_ptr() for f in ptrs} == ptrs
    for f in ("rowptr_dst", "rowptr_src"):
        assert torch.equal(getattr(ca, f), getattr(fresh, f)), f
    for f in ("edge_src", "edge_dst", "eid_coo", "src_eid"):
        assert torch.equal(getattr(ca, f)[:E2], getattr(fresh, f)), f
    s_src, s_dst = ops.src_sorted_pairs(fresh)
    assert torch.equal(ca.s_src[:E2], s_src) and torch.equal(ca.s_dst[:E2], s_dst)
    # consumers that visit all n_edges rows refuse a capacity set
    with pytest.raises(ValueError, match="exact-size"):
        ops.require_exact(ca, "test")


def _obs(cfg_name, B, seed):
    cfg = CONFIGS[cfg_name]
    gen = torch.Generator().manual_seed(seed)
    return cfg, synthetic_obs(cfg, B, gen, env_ids=torch.arange(B) * max(1, cfg.num_envs // B) % cfg.num_envs)


def _radius_data(cfg, refresh: bool, radius=None):
    """The policy graph's data builder (tests/gpu_helpers.make_data) with radius INTERNAL edges, feeding HEPi."""
    from geometry_rl_b200.synthetic import observation_layout
    r, m = RADIUS[cfg.name]
    r = r if radius is None else radius
    D = type(G.make_data(cfg, policy=True))
    dims, names = observation_layout(cfg)
    data = D(observation_dim=dims, observation_names=names, full_graph_obs=False, dist_as_pos=True,
             output_mask_key="grippers", concat_input_vector=False, angular_velocity=cfg.angular_velocity,
             internal_edges="radius", radius=r, max_num_neighbors=m)
    data.consumer_accepts_capacity = True
    data.rebuild_every_call = refresh
    return data


def _oracle_topology(cfg, obs):
    from oracle import graph as og
    from tests.radius_oracle import radius_topology
    from geometry_rl_b200.synthetic import observation_layout, obs_keys
    r, m = RADIUS[cfg.name]
    dims, names = observation_layout(cfg)
    parts = og.split_obs({k: obs[k] for k in obs_keys(cfg)}, dims, names)
    num_points = parts["infos"]["object_num_points"].long().reshape(-1) if cfg.task == "rigid" else None
    return radius_topology(og.TASKS[cfg.task], parts["position_vectors"], full_graph_obs=False,
                           output_mask_key="grippers", num_points=num_points, radius=r, max_num_neighbors=m)


def _assert_topology(graph, og_graph):
    for et in og_graph.edge_types:
        es = graph.edge_sets[et]
        E = int(es.edge_ptr[-1])
        assert torch.equal(es.coo[:, :E].cpu(), og_graph.edge_index_dict[et]), f"COO {et}"
        assert torch.equal((es.edge_ptr[1:] - es.edge_ptr[:-1]).cpu(), og_graph.edge_counts[et]), f"edge_ptr {et}"
        if not es.exact:
            assert not bool(es.coo[:, E:].any()) and int(es.rowptr_dst[-1]) == E


@pytest.mark.parametrize("cfg_name", [ROPE, RIGID])
def test_data_builders_give_the_oracle_radius_topology(cfg_name, sixteen_bit):
    for refresh in (False, True):
        cfg, obs0 = _obs(cfg_name, 9, 11)
        _, obs1 = _obs(cfg_name, 9, 12)
        data = _radius_data(cfg, refresh)
        assert data.refresh_in_place() == refresh
        g0, _ = data.build_data(*G.obs_args(cfg, obs0, policy=True), train=False)
        _assert_topology(g0, _oracle_topology(cfg, obs0))
        g1, _ = data.build_data(*G.obs_args(cfg, obs1, policy=True), train=False)
        # build-once keeps the first batch's topology; refresh mode follows the positions of this call, in place
        _assert_topology(g1, _oracle_topology(cfg, obs1 if refresh else obs0))
        if refresh:
            et = ("links", "internal", "links") if cfg.task == "rope" else ("object_geometry", "internal", "object_geometry")
            assert g1.edge_sets[et] is g0.edge_sets[et] and not g1.edge_sets[et].exact
            assert (et[0], "task", "grippers") in g1.refreshed_edge_types or cfg.task == "rope"


def _agent(cfg_name, B, seed=0, refresh=False):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    cfg = CONFIGS[cfg_name]
    actor, critic, projection, loss_module, adv_module = learner.build_agent(cfg, G.dev(), seed=seed)
    hd = actor.get_submodule("0").module.hyper_data
    r, m = RADIUS[cfg_name]
    hd.internal_edges, hd.radius, hd.max_num_neighbors = "radius", r, m
    hd.rebuild_every_call = refresh
    gen = torch.Generator().manual_seed(199 + seed)
    obs = synthetic_obs(cfg, B, gen, env_ids=torch.arange(B) * max(1, cfg.num_envs // B) % cfg.num_envs)
    with torch.no_grad():
        actor.get_dist(to_device(obs, G.dev()))
        for n, p in actor.named_parameters():
            if n.endswith("bias") and float(p.abs().max()) == 0:
                p.normal_(0, 0.05)
    return cfg, actor, critic, loss_module, obs, gen, hd


def _oracle_step(cfg, actor, critic, mb):
    """Oracle losses and gradients of one step from the current parameters, on the radius topology of `mb`."""
    from oracle.step import OracleAgent
    oracle = OracleAgent(cfg, actor.state_dict(), critic.state_dict())
    B = mb["scalars"].shape[0]
    oracle._topo[True] = {B: _oracle_topology(cfg, mb)}  # the radius topology of THIS minibatch
    return oracle.step_grads(mb)


@pytest.mark.parametrize("cfg_name,refresh", [(ROPE, False), (ROPE, True), (RIGID, True)])
def test_16bit_update_step_on_radius_topology_matches_oracle(cfg_name, refresh, sixteen_bit):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    from oracle.step import OracleAgent, make_minibatch
    from tests.test_gpu_step16 import _compare
    cfg, actor, critic, loss_module, obs, gen, hd = _agent(cfg_name, 6 if cfg_name == ROPE else 24, refresh=refresh)
    mb = make_minibatch(cfg, OracleAgent(cfg, actor.state_dict(), critic.state_dict()), obs, gen)
    ref, ga, gc = _oracle_step(cfg, actor, critic, mb)
    lrn = learner.Learner(cfg, actor, critic, loss_module)
    out = lrn.compute_losses(to_device(mb, G.dev()))
    out["actor_loss"].backward()
    out["loss_critic"].backward()
    assert hd.refresh_in_place() == refresh
    pol = {k: p.grad for k, p in actor.get_submodule("0").module.named_parameters()}
    vf = {k: p.grad for k, p in critic.module._network1.named_parameters()}
    report = []
    bad = _compare(out, ref, pol, ga, vf, gc, report)
    assert not bad, "\n".join(bad + ["--"] + report)


def test_captured_replay_rebuilds_the_radius_graph_every_step(sixteen_bit):
    """Capture on minibatch A, replay B and C (moved positions): after each replay the graph's edge sets are the oracle
    radius graph of that minibatch; losses and gradients equal the eager refresh-mode `update` from the same state
    (bit-identical) and the oracle (1e-2)."""
    import dataclasses
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    from oracle.step import OracleAgent, make_minibatch
    from tests.test_gpu_step16 import _compare
    B = 8
    runs = {}
    for mode in ("graphed", "eager"):
        cfg, actor, critic, loss_module, obs, gen, hd = _agent(ROPE, B, seed=3, refresh=True)
        o0 = OracleAgent(cfg, actor.state_dict(), critic.state_dict())
        mbs = []
        for s in range(3):
            _, o = _obs(ROPE, B, 40 + s)  # the rope moves from minibatch to minibatch
            mbs.append(make_minibatch(cfg, o0, o, gen))
        # no gradient clipping: the flat bucket then holds the gradients the oracle computes
        lrn = learner.Learner(dataclasses.replace(cfg, clip_grad_norm=False), actor, critic, loss_module,
                              overlap_critic=False)
        res = []
        if mode == "graphed":
            lrn.capture(to_device(mbs[0], G.dev()), warmup=2)
        for mb in mbs[1:]:
            ref = _oracle_step(cfg, actor, critic, mb)
            out = lrn.update_graphed(to_device(mb, G.dev())) if mode == "graphed" else lrn.update(to_device(mb, G.dev()))
            torch.cuda.synchronize()
            _assert_topology(hd.example_data, _oracle_topology(cfg, mb))
            flat = {k: v.clone() for k, v in lrn.flat_grads().items()}
            res.append(({k: float(out[k]) for k in ("loss_objective", "loss_critic", "kl", "entropy")}, flat))
            pol = {k[len("actor.0.module."):]: v for k, v in flat.items() if k.startswith("actor.0.module.")}
            vf = {k[len("critic.module._network1."):]: v for k, v in flat.items() if k.startswith("critic.module._network1.")}
            report = []
            bad = _compare(out, ref[0], pol, ref[1], vf, ref[2], report)
            assert not bad, "\n".join([mode] + bad + ["--"] + report)
        runs[mode] = res
    for (lg, fg), (le, fe) in zip(runs["graphed"], runs["eager"]):
        assert lg == le
        for k in fg:
            assert torch.equal(fg[k], fe[k]), k


def test_pruned_rows_equal_dense_in_refresh_mode(sixteen_bit):
    from geometry_rl_b200 import ops
    cfg, obs0 = _obs(ROPE, 10, 21)
    _, obs1 = _obs(ROPE, 10, 22)
    torch.manual_seed(5)
    net = G.make_policy_body(cfg)
    with torch.no_grad():
        for n, p in net.named_parameters():
            if n.endswith("bias") and float(p.abs().max()) == 0:
                p.normal_(0, 0.05)
    net.eval()
    data = _radius_data(cfg, refresh=True)
    data.build_data(*G.obs_args(cfg, obs0, policy=True), train=False)
    graph, u = data.build_data(*G.obs_args(cfg, obs1, policy=True), train=False)  # refreshed in place
    pr = graph.hetero_pruned()
    assert "target_geometry" not in pr.live_ids
    et = ("links", "internal", "links")
    assert pr.edge_sets[et] is graph.edge_sets[et]
    gen = torch.Generator().manual_seed(2)
    res = {}
    for prune in (False, True):
        net.prune_dead_rows = prune
        net.zero_grad(set_to_none=True)
        out, hidden = net.one_step(graph, u)
        if not prune:
            w_out = torch.randn(out.shape, generator=gen).cuda()
            w_hid = torch.randn(hidden.shape, generator=gen).cuda()
        loss = (out * w_out).sum() + (hidden * w_hid).sum()
        n_e = sum(es.n_edges for es in graph.edge_sets.values())
        for numel, dt in ((n_e * 1024, torch.bfloat16), (n_e * 1024, torch.float32), (graph.num_nodes * 1024, torch.float32)):
            for frac in (1.0, 0.5, 0.25):
                junk = torch.full((max(1, int(numel * frac)),), float("nan"), dtype=dt, device="cuda")
                del junk
        loss.backward()
        res[prune] = (out.detach().clone(), hidden.detach().clone(),
                      {k: p.grad.detach().clone() for k, p in net.named_parameters() if p.grad is not None})
    (o0, h0, g0), (o1, h1, g1) = res[False], res[True]
    assert G.rel(o1, o0) < 4e-3, G.err_report("out", o1, o0)
    assert G.rel(h1, h0) < 4e-3, G.err_report("hidden", h1, h0)
    assert set(g0) == set(g1)
    for k in g0:
        assert G.rel(g1[k], g0[k]) < 4e-3, G.err_report(k, g1[k], g0[k])


def test_calibration_identical_with_capacity_and_exact_topology(sixteen_bit):
    cfg, obs = _obs(ROPE, 12, 31)
    factors = {}
    for refresh in (False, True):
        torch.manual_seed(7)
        net = G.make_policy_body(cfg)
        net.train()
        data = _radius_data(cfg, refresh)
        graph, u = data.build_data(*G.obs_args(cfg, obs, policy=True), train=False)
        assert any(not es.exact for es in graph.edge_sets.values()) == refresh
        with torch.no_grad():
            net.one_step(graph, u)
        factors[refresh] = {k: v.detach().clone() for k, v in net.state_dict().items()}
    for k, v in factors[False].items():
        assert torch.equal(factors[True][k], v), k


def test_all_empty_radius_batch(sixteen_bit):
    """No INTERNAL edge in the whole batch (a radius below every link spacing).  Exact topology skips the edge type (as
    the reference does); fixed-capacity topology runs the convolution with empty neighbourhoods
    (BaseData._refresh_topology), so a sample gets the output it gets next to samples that have edges."""
    cfg, obs = _obs(ROPE, 6, 51)
    torch.manual_seed(9)
    net = G.make_policy_body(cfg)
    with torch.no_grad():
        for n, p in net.named_parameters():
            if n.endswith("bias") and float(p.abs().max()) == 0:
                p.normal_(0, 0.05)
    net.eval()
    et = ("links", "internal", "links")
    tiny = 1e-3  # the closest links of this batch are 1.4e-3 apart
    data = _radius_data(cfg, True, radius=tiny)
    graph, u = data.build_data(*G.obs_args(cfg, obs, policy=True), train=False)
    assert int(graph.edge_sets[et].rowptr_dst[-1]) == 0 and graph.edge_sets[et].n_edges > 0
    out_empty, hidden = net.one_step(graph, u)
    assert bool(torch.isfinite(out_empty).all()) and bool(torch.isfinite(hidden).all())
    # exact topology of the same batch: the edge type is empty and its convolution is skipped
    data_x = _radius_data(cfg, False, radius=tiny)
    graph_x, u_x = data_x.build_data(*G.obs_args(cfg, obs, policy=True), train=False)
    assert graph_x.edge_sets[et].n_edges == 0
    out_x, _ = net.one_step(graph_x, u_x)
    assert bool(torch.isfinite(out_x).all())
    # samples 1.. get one pair of links within the radius; sample 0 keeps no INTERNAL edge and its output is unchanged
    mixed = {k: v.clone() for k, v in obs.items()}
    names = [str(n) for n in data.observation_names["position_vectors"]]
    off = sum(data.observation_dim["position_vectors"][: names.index("links")])
    mixed["position_vectors"][1:, off + 3:off + 6] = mixed["position_vectors"][1:, off:off + 3] + 1e-4
    graph_m, u_m = data.build_data(*G.obs_args(cfg, mixed, policy=True), train=False)
    assert graph_m.edge_sets[et] is graph.edge_sets[et]
    counts = (graph_m.edge_sets[et].edge_ptr[1:] - graph_m.edge_sets[et].edge_ptr[:-1]).cpu()
    assert counts.tolist() == [0, 2, 2, 2, 2, 2]
    out_m, _ = net.one_step(graph_m, u_m)
    A = out_m.shape[0] // 6
    assert G.rel(out_m[:A], out_empty[:A]) < 1e-5, G.err_report("sample 0", out_m[:A], out_empty[:A])


def test_capture_refuses_eager_rebuild_modes():
    from geometry_rl_b200 import learner, ops
    from geometry_rl_b200.tensors import to_device
    for internal, precision in (("knn", "bf16"), ("radius", "fp32")):
        ops.set_precision(precision)
        try:
            cfg, actor, critic, loss_module, obs, gen, hd = _agent(ROPE, 4, refresh=False)
            if internal == "knn":
                hd.internal_edges, hd.radius = "knn", None
            hd.rebuild_every_call = True
            lrn = learner.Learner(cfg, actor, critic, loss_module)
            with pytest.raises(ValueError, match="cannot be replayed"):
                lrn.capture({k: v for k, v in to_device(obs, G.dev()).items()})
            assert lrn._graph is None
        finally:
            ops.set_precision("fp32")
