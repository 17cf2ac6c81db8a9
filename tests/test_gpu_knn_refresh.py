"""GPU: kNN topology written in one pass (grl_knn_topology, ops.knn_edge_set) and rebuilt in place on every call
(`rebuild_every_call` + `knn_in_place`), inside the captured update and the acting graph.

Integer topology is compared with torch.equal against today's chain (knn_graph -> build_edge_set -> src_sorted_pairs)
and the numpy restatement (tests/knn_topology_reference.py).  Rope has no padded rows and its in-place set is exact-size,
so the strict fp32 update replayed from a CUDA graph is bit-identical to the eager rebuild; 16-bit steps are held to
north_star's bound (1e-2 of each tensor's max magnitude) against the oracle, as in test_gpu_radius.py."""
import dataclasses
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from geometry_rl_b200.synthetic import CONFIGS, synthetic_obs
from tests import gpu_helpers as G
from tests.knn_topology_reference import one_pass_layouts

pytestmark = pytest.mark.gpu

ROPE, RIGID = "rope_shaping_hepi_trpl_cfg", "rigid_insertion_multi_hepi_trpl_cfg"
FIELDS = ("coo", "edge_ptr", "rowptr_dst", "edge_src", "edge_dst", "eid_coo", "rowptr_src", "src_eid", "s_src", "s_dst")


@pytest.fixture
def sixteen_bit():
    from geometry_rl_b200 import ops
    ops.set_precision("bf16")
    yield
    ops.set_precision("fp32")


def _chain(pos, nv, k, capacity=None):
    """Today's path: knn_graph -> build_edge_set (exact, or a zero-padded capacity COO) -> src_sorted_pairs."""
    from geometry_rl_b200 import ops
    B, P, _ = pos.shape
    coo, ptr = ops.knn_graph(pos, nv, k)
    if capacity is None:
        es = ops.build_edge_set(coo, ptr, B, P, P)
    else:
        buf = torch.zeros(2, capacity, dtype=torch.int64, device=pos.device)
        buf[:, :coo.shape[1]] = coo
        es = ops.build_edge_set(buf, ptr, B, P, P, exact=False)
    ops.src_sorted_pairs(es)
    return es


def _assert_same(a, b, what):
    assert (a.n_src, a.n_dst, a.n_edges, a.exact) == (b.n_src, b.n_dst, b.n_edges, b.exact), what
    for f in FIELDS:
        x, y = getattr(a, f), getattr(b, f)
        assert x.dtype == y.dtype and x.shape == y.shape, (what, f, x.shape, y.shape)
        assert torch.equal(x, y), (what, f)


def _positions(B, P, seed, rope=False):
    gen = torch.Generator().manual_seed(seed)
    if rope:  # a chain of links ~0.01 apart, as the rope observations
        return torch.cumsum(torch.randn(B, P, 3, generator=gen) * 0.01, dim=1).cuda()
    return (torch.rand(B, P, 3, generator=gen) * 0.3).cuda()


def _num_valid(B, P, seed):
    gen = torch.Generator().manual_seed(seed)
    nv = torch.randint(0, P + 1, (B,), generator=gen, dtype=torch.int32)
    nv[:4] = torch.tensor([0, 1, 2, 3], dtype=torch.int32)[: min(4, B)]
    nv[-1] = P
    return nv.cuda()


@pytest.mark.parametrize("B", [1, 37, 2048])
def test_rope_shapes_kernel_equals_chain(B):
    from geometry_rl_b200 import ops
    P, k = 80, 3
    pos = _positions(B, P, B, rope=True)
    _assert_same(ops.knn_edge_set(pos, None, k), _chain(pos, None, k), "exact")
    _assert_same(ops.knn_edge_set(pos, None, k, capacity=B * P * k), _chain(pos, None, k, B * P * k), "capacity")


@pytest.mark.parametrize("B,P,k", [(7, 48, 3), (512, 48, 3), (8192, 48, 3), (33, 512, 8), (64, 9, 8), (16, 2, 3)])
def test_rigid_shapes_kernel_equals_chain(B, P, k):
    from geometry_rl_b200 import ops
    pos, nv = _positions(B, P, 11 + B), _num_valid(B, P, 5 + P)
    es = ops.knn_edge_set(pos, nv, k)
    assert not es.exact and es.n_edges == B * P * k
    _assert_same(es, _chain(pos, nv, k, B * P * k), "capacity")
    if B <= 64:
        ref = one_pass_layouts(pos.cpu().numpy(), nv.cpu().numpy(), k, B * P * k)
        for f in FIELDS:
            assert np.array_equal(getattr(es, f).cpu().numpy(), ref[f]), f


def test_all_graphs_without_edges():
    from geometry_rl_b200 import ops
    pos, nv = _positions(5, 12, 1), torch.tensor([0, 1, 1, 0, 1], dtype=torch.int32, device="cuda")
    es = ops.knn_edge_set(pos, nv, 3)
    _assert_same(es, _chain(pos, nv, 3, 5 * 12 * 3), "empty")
    assert int(es.edge_ptr[-1]) == 0 and not bool(es.edge_dst.any()) and not bool(es.s_src.any())
    one = ops.knn_edge_set(_positions(4, 1, 2), None, 3)  # P = 1: an exact set of no edges
    _assert_same(one, _chain(_positions(4, 1, 2), None, 3), "P=1")


def test_non_finite_positions():
    """NaN / inf points: exactly edge_ptr edges, indices in bounds, the same result on a repeat, and the finite graphs
    equal to a build without the bad points."""
    from geometry_rl_b200 import ops
    B, P, k = 12, 48, 3
    pos, nv = _positions(B, P, 3), _num_valid(B, P, 4)
    nv[5:9] = P
    bad = pos.clone()
    bad[5, 7, 1] = float("nan")
    bad[6] = float("nan")
    bad[7, 0] = float("inf")
    bad[8, 3, 2] = -float("inf")
    bad_graphs = [5, 6, 7, 8]
    for nv_, cap in ((nv, B * P * k), (None, None)):
        es = ops.knn_edge_set(bad, nv_, k, capacity=cap)
        torch.cuda.synchronize()
        E = int(es.edge_ptr[-1])
        assert int(es.rowptr_dst[-1]) == E == int(es.rowptr_src[-1])
        counts = (es.rowptr_dst[1:] - es.rowptr_dst[:-1]).cpu()
        assert int(counts.sum()) == E and bool((counts >= 0).all())
        for f in ("edge_src", "edge_dst", "s_src", "s_dst"):
            t = getattr(es, f)
            assert bool((t >= 0).all() and (t < B * P).all()), f
        for f in ("eid_coo", "src_eid"):
            t = getattr(es, f)[:E]
            assert torch.equal(torch.sort(t.long()).values, torch.arange(E, device="cuda")), f
        again = ops.knn_edge_set(bad, nv_, k, capacity=cap)
        _assert_same(again, es, "repeat")
        ref = one_pass_layouts(bad.cpu().numpy(), None if nv_ is None else nv_.cpu().numpy(), k, es.n_edges)
        for f in FIELDS:
            assert np.array_equal(getattr(es, f).cpu().numpy(), ref[f]), f
        clean = ops.knn_edge_set(pos, nv_, k, capacity=cap)
        for g in range(B):
            if g in bad_graphs:
                continue
            e0, e1 = int(es.edge_ptr[g]), int(es.edge_ptr[g + 1])
            for f in ("edge_src", "edge_dst", "eid_coo", "src_eid", "s_src", "s_dst"):
                assert torch.equal(getattr(es, f)[e0:e1], getattr(clean, f)[e0:e1]), (g, f)
            assert torch.equal(es.coo[:, e0:e1], clean.coo[:, e0:e1]), g
            assert torch.equal(es.rowptr_dst[g * P:(g + 1) * P], clean.rowptr_dst[g * P:(g + 1) * P]), g
            assert torch.equal(es.rowptr_src[g * P:(g + 1) * P], clean.rowptr_src[g * P:(g + 1) * P]), g


@pytest.mark.parametrize("rigid", [False, True])
def test_captured_refresh_follows_new_positions(rigid):
    from geometry_rl_b200 import ops
    B, P, k = (96, 48, 3) if rigid else (64, 80, 3)
    pos = _positions(B, P, 21, rope=not rigid)
    nv = _num_valid(B, P, 22) if rigid else None
    es = ops.knn_edge_set(pos, nv, k)
    ptrs = {f: getattr(es, f).data_ptr() for f in FIELDS}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.refresh_knn_edge_set(es, pos, nv, k)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.refresh_knn_edge_set(es, pos, nv, k)
    for seed in (23, 24):
        pos.copy_(_positions(B, P, seed, rope=not rigid))
        if rigid:
            nv.copy_(_num_valid(B, P, seed))
        g.replay()
        torch.cuda.synchronize()
        assert {f: getattr(es, f).data_ptr() for f in FIELDS} == ptrs
        _assert_same(es, ops.knn_edge_set(pos, nv, k), f"replay {seed}")
        _assert_same(es, _chain(pos, nv, k, None if nv is None else B * P * k), f"chain {seed}")


def test_data_builders_refresh_the_knn_set_in_place(sixteen_bit):
    from oracle import graph as og
    from geometry_rl_b200.synthetic import observation_layout, obs_keys
    for cfg_name in (ROPE, RIGID):
        cfg, obs0 = _obs(cfg_name, 9, 11)
        _, obs1 = _obs(cfg_name, 9, 12)
        data = G.make_data(cfg, policy=True)
        data.consumer_accepts_capacity, data.rebuild_every_call, data.knn_in_place = True, True, True
        assert data.refresh_in_place()
        g0, _ = data.build_data(*G.obs_args(cfg, obs0, policy=True), train=False)
        g1, _ = data.build_data(*G.obs_args(cfg, obs1, policy=True), train=False)
        et = (data.PARTICLE_TYPE, "internal", data.PARTICLE_TYPE)
        es = g1.edge_sets[et]
        assert es is g0.edge_sets[et] and et in g1.refreshed_edge_types and es.exact == (cfg.task == "rope")
        dims, names = observation_layout(cfg)
        parts = og.split_obs({k: obs1[k] for k in obs_keys(cfg)}, dims, names)
        num_points = parts["infos"]["object_num_points"].long().reshape(-1) if cfg.task == "rigid" else None
        ref = og.build_topology(og.TASKS[cfg.task], parts["position_vectors"], full_graph_obs=False,
                                output_mask_key="grippers", num_points=num_points)
        for t in ref.edge_types:
            E = int(g1.edge_sets[t].edge_ptr[-1])
            assert torch.equal(g1.edge_sets[t].coo[:, :E].cpu(), ref.edge_index_dict[t]), t


def _obs(cfg_name, B, seed):
    cfg = CONFIGS[cfg_name]
    gen = torch.Generator().manual_seed(seed)
    return cfg, synthetic_obs(cfg, B, gen, env_ids=torch.arange(B) * max(1, cfg.num_envs // B) % cfg.num_envs)


def _agent(cfg_name, B, seed=0, in_place=True):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    cfg = CONFIGS[cfg_name]
    actor, critic, projection, loss_module, adv_module = learner.build_agent(cfg, G.dev(), seed=seed)
    hd = actor.get_submodule("0").module.hyper_data
    hd.rebuild_every_call, hd.knn_in_place = True, in_place
    gen = torch.Generator().manual_seed(199 + seed)
    obs = synthetic_obs(cfg, B, gen, env_ids=torch.arange(B) * max(1, cfg.num_envs // B) % cfg.num_envs)
    with torch.no_grad():
        actor.get_dist(to_device(obs, G.dev()))
        for n, p in actor.named_parameters():
            if n.endswith("bias") and float(p.abs().max()) == 0:
                p.normal_(0, 0.05)
    return cfg, actor, critic, loss_module, obs, gen, hd


def _oracle_step(cfg, actor, critic, mb):
    """Oracle losses and gradients of one step from the current parameters, on the kNN topology of `mb`."""
    from oracle import graph as og
    from oracle.step import OracleAgent
    from geometry_rl_b200.synthetic import observation_layout, obs_keys
    oracle = OracleAgent(cfg, actor.state_dict(), critic.state_dict())
    dims, names = observation_layout(cfg)
    parts = og.split_obs({k: mb[k] for k in obs_keys(cfg)}, dims, names)
    num_points = parts["infos"]["object_num_points"].long().reshape(-1) if cfg.task == "rigid" else None
    B = mb["scalars"].shape[0]
    oracle._topo[True] = {B: og.build_topology(og.TASKS[cfg.task], parts["position_vectors"], full_graph_obs=False,
                                               output_mask_key="grippers", num_points=num_points)}
    return oracle.step_grads(mb)


def _run(cfg_name, B, mode, n=3):
    """`n - 1` updates after capturing on minibatch 0: 'graphed' (in-place kNN, replayed), 'eager_in_place' (the same
    rebuild, `update`), 'eager' (today's eager exact-size rebuild, `update`).  Returns (losses, flat grads, params,
    oracle results) per step."""
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    from oracle.step import OracleAgent, make_minibatch
    cfg, actor, critic, loss_module, obs, gen, hd = _agent(cfg_name, B, seed=3, in_place=mode != "eager")
    assert hd.refresh_in_place() == (mode != "eager")
    o0 = OracleAgent(cfg, actor.state_dict(), critic.state_dict())
    mbs = [make_minibatch(cfg, o0, _obs(cfg_name, B, 40 + s)[1], gen) for s in range(n)]  # the positions move
    lrn = learner.Learner(dataclasses.replace(cfg, clip_grad_norm=False), actor, critic, loss_module,
                          overlap_critic=False)
    if mode == "graphed":
        lrn.capture(to_device(mbs[0], G.dev()), warmup=2)
    res = []
    for mb in mbs[1:]:
        ref = _oracle_step(cfg, actor, critic, mb) if mode == "graphed" else None
        out = lrn.update_graphed(to_device(mb, G.dev())) if mode == "graphed" else lrn.update(to_device(mb, G.dev()))
        torch.cuda.synchronize()
        out = {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in out.items()}  # replay outputs are static
        res.append(({k: float(out[k]) for k in ("loss_objective", "loss_critic", "kl", "entropy")},
                    {k: v.clone() for k, v in lrn.flat_grads().items()},
                    {k: p.detach().clone() for k, p in list(actor.named_parameters()) + list(critic.named_parameters())},
                    (out, ref)))
    return res


def test_captured_fp32_rope_update_is_bit_identical_to_the_eager_rebuild():
    graphed, eager = _run(ROPE, 8, "graphed"), _run(ROPE, 8, "eager")
    for (lg, fg, pg, _), (le, fe, pe, _) in zip(graphed, eager):
        assert lg == le
        for k in fe:
            assert torch.equal(fg[k], fe[k]), k
        for k in pe:
            assert torch.equal(pg[k], pe[k]), k


@pytest.mark.parametrize("cfg_name,B", [(ROPE, 8), (RIGID, 24)])
def test_captured_16bit_update_matches_oracle_and_eager(cfg_name, B, sixteen_bit):
    from tests.test_gpu_step16 import _compare
    graphed, eager = _run(cfg_name, B, "graphed"), _run(cfg_name, B, "eager_in_place")
    for (lg, fg, _, (out, ref)), (le, fe, _, _) in zip(graphed, eager):
        pol = {k[len("actor.0.module."):]: v for k, v in fg.items() if k.startswith("actor.0.module.")}
        vf = {k[len("critic.module._network1."):]: v for k, v in fg.items() if k.startswith("critic.module._network1.")}
        report = []
        bad = _compare(out, ref[0], pol, ref[1], vf, ref[2], report)
        assert not bad, "\n".join(bad + ["--"] + report)
        assert lg == le  # the same in-place rebuild replayed or launched eagerly
        for k in fe:
            assert torch.equal(fg[k], fe[k]), k


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_act_graph_with_in_place_knn_follows_the_positions(precision):
    """capture_act + act_graphed == eager act on the same positions and Philox state; act replays interleaved with
    captured update replays leave both correct."""
    from geometry_rl_b200 import learner, ops
    from geometry_rl_b200.tensors import to_device
    from tests.test_gpu_act import _obs_batches, _outs
    ops.set_precision(precision)
    try:
        cfg, actor, critic, loss_module, obs, gen, hd = _agent(ROPE, 6, seed=4)
        assert hd.refresh_in_place()
        batches = _obs_batches(cfg, 6, 4, 900)  # the rope moves from batch to batch
        actor.capture_act(batches[0], seed=31)
        lrn = learner.Learner(cfg, actor, critic, loss_module)
        from oracle.step import OracleAgent, make_minibatch
        mb = to_device(make_minibatch(cfg, OracleAgent(cfg, actor.state_dict(), critic.state_dict()), obs, gen), G.dev())
        lrn.capture(mb, warmup=2)
        graphed = []
        for i, td in enumerate(batches[1:]):
            state = actor.act_state()
            replayed, eager = dict(td), dict(td)
            actor.act_graphed(replayed)
            actor.set_act_state(*state)
            actor.act(eager)  # same positions, same Philox state, the parameters the replay read
            for got, exp in zip(_outs(replayed), _outs(eager)):
                assert torch.equal(got, exp), i
            graphed.append(_outs(replayed))
            lrn.update_graphed(mb)  # the update graph rewrites the shared placeholder from its own positions
        assert not torch.equal(graphed[0][0], graphed[1][0])
    finally:
        ops.set_precision("fp32")


def test_capture_guards():
    """Refused with the flag: rigid on the strict fp32 path (its kNN set would need a capacity) and EMPN (homogeneous
    view).  kNN without the flag is refused by test_gpu_radius.py / test_gpu_act.py, unchanged."""
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    from tests.test_gpu_act import _obs_batches
    for cfg_name in (RIGID, "rigid_pushing_multi_empn_trpl_cfg"):
        cfg = CONFIGS[cfg_name]
        actor, critic, _, loss_module, _ = learner.build_agent(cfg, G.dev(), seed=0)
        hd = actor.get_submodule("0").module.hyper_data
        hd.rebuild_every_call, hd.knn_in_place = True, True
        assert not hd.refresh_in_place()
        obs = _obs_batches(cfg, 4, 1, 5)[0]
        lrn = learner.Learner(cfg, actor, critic, loss_module)
        with pytest.raises(ValueError, match="cannot be replayed"):
            lrn.capture({k: v for k, v in to_device(obs, G.dev()).items()})
        with pytest.raises(ValueError, match="cannot be replayed"):
            actor.capture_act(obs, seed=0)


# ---- two ranks, each rebuilding the kNN set of its half of the minibatch (gloo rendezvous, as test_gpu_radius_dp.py)
DP_B = 8
DP_KEYS = ("loss_objective", "loss_critic", "kl", "entropy")


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_setup(dev):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    from geometry_rl_b200.synthetic import synthetic_minibatch
    cfg = CONFIGS[ROPE]
    actor, critic, _, loss_module, _ = learner.build_agent(cfg, dev, seed=0)
    hd = actor.get_submodule("0").module.hyper_data
    hd.rebuild_every_call, hd.knn_in_place = True, True
    assert hd.refresh_in_place()
    gen = torch.Generator().manual_seed(78)
    obs = synthetic_obs(cfg, DP_B, gen, env_ids=torch.arange(DP_B) * (cfg.num_envs // DP_B))
    with torch.no_grad():  # calibration on the FULL batch in every process -> identical replicas
        d = actor.get_dist(to_device(obs, dev))
        v = critic.module(*[obs[k].to(dev) for k in critic.in_keys])
    return cfg, actor, critic, loss_module, synthetic_minibatch(obs, d.mean, d.var_diag, v, gen)


def _grads(actor, critic):
    return [p.grad.detach().cpu().clone() if p.grad is not None else None
            for p in list(actor.parameters()) + list(critic.parameters())]


def _dp_worker(rank, world, port, out_path):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from geometry_rl_b200 import learner
        from geometry_rl_b200.parallel import DataParallel
        from geometry_rl_b200.tensors import to_device
        dev = torch.device("cuda", rank if torch.cuda.device_count() >= world else 0)
        torch.cuda.set_device(dev)
        cfg, actor, critic, loss_module, mb = _dp_setup(dev)
        dp = DataParallel()
        lrn = learner.Learner(cfg, actor, critic, loss_module, dp=dp)
        sl = slice(rank * DP_B // world, (rank + 1) * DP_B // world)
        out = lrn.compute_losses(to_device({k: (v[sl] if torch.is_tensor(v) else v) for k, v in mb.items()}, dev))
        out["actor_loss"].backward()
        out["loss_critic"].backward()
        dp.allreduce_grads(list(actor.parameters()) + list(critic.parameters()))
        logged = dp.global_losses(out)
        torch.cuda.synchronize()
        if rank == 0:
            torch.save({"losses": {k: logged[k].detach().cpu() for k in DP_KEYS}, "grads": _grads(actor, critic)},
                       out_path)
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_rank_step_with_in_place_knn_equals_single_process(tmp_path):
    """fp32, one rank per GPU (both on one GPU when there is only one): losses and all-reduced gradients equal the
    single-process step within 1e-4."""
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    world, port = 2, _free_port()
    out_path = str(tmp_path / "rank0.pt")
    procs = [mp.get_context("spawn").Process(target=_dp_worker, args=(r, world, port, out_path)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    res = torch.load(out_path, weights_only=True)
    dev = torch.device("cuda:0")
    cfg, actor, critic, loss_module, mb = _dp_setup(dev)
    out = learner.Learner(cfg, actor, critic, loss_module).compute_losses(to_device(mb, dev))
    out["actor_loss"].backward()
    out["loss_critic"].backward()
    for k in DP_KEYS:
        a, b = float(res["losses"][k]), float(out[k])
        assert abs(a - b) <= 1e-4 * max(1.0, abs(b)), (k, a, b)
    for i, (g_dp, g1) in enumerate(zip(res["grads"], _grads(actor, critic))):
        if g1 is None or float(g1.abs().max()) == 0.0:
            continue
        assert float((g_dp - g1).abs().max()) <= 1e-4 * float(g1.abs().max()), i
