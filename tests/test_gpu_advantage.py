"""GPU: the advantage phase on the fused critic kernels (GAE.advantage / capture / advantage_graphed / advantage_static).
The grouped grl_critic_inner_stats + _fwd against an fp64 restatement of per-group LayerNorm(mode='graph'); GAE.advantage
against the oracle's per-step critic loop + reverse GAE for the five configs and against `adv_module(td)`; replays
bit-identical to eager calls, interleaved with captured update and act replays; two ranks holding half the environments
each against one process; the capture guard."""
import ctypes as C
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

from geometry_rl_b200.synthetic import CONFIGS, CONFIG_ORDER, synthetic_rollout
from tests import gpu_helpers as G

pytestmark = pytest.mark.gpu

RIGID, CLOTH = "rigid_insertion_multi_hepi_trpl_cfg", "cloth_hanging_multi_hepi_trpl_cfg"
OUT_KEYS = ("advantage", "value_target", "state_value")


# ---- 1. the grouped kernels alone ------------------------------------------------------------------------------------
def _grouped_ref(x, p, groups, eps):
    D = torch.float64
    h = F.linear(x.to(D), p["w1"].to(D), p["b1"].to(D))  # [B, N, 64]
    hg = h.reshape(groups, -1)
    mean = hg.mean(1, keepdim=True)
    std = (hg - mean).pow(2).mean(1, keepdim=True).sqrt()
    xh = ((hg - mean) / (std + eps)).reshape(h.shape)
    return torch.relu(xh * p["gamma"].to(D) + p["beta"].to(D)).sum(1), torch.cat([hg.sum(1, keepdim=True),
                                                                                   hg.pow(2).sum(1, keepdim=True)], 1)


@pytest.mark.parametrize("b_env,groups,N,Fd", [(64, 1, 97, 15), (1, 2, 97, 15), (3, 101, 97, 15), (5, 4, 300, 16),
                                               (2, 300, 40, 13), (7, 17, 239, 12)])
def test_grouped_kernel_matches_fp64(b_env, groups, N, Fd):
    from geometry_rl_b200 import _lib as L
    from geometry_rl_b200 import ops
    B = b_env * groups
    g = torch.Generator().manual_seed(B * 7 + N)
    r = lambda *s, scale=1.0: (torch.randn(*s, generator=g) * scale).cuda()
    # a per-group offset, so that statistics shared across groups would be visibly wrong
    x = (r(groups, b_env, N, Fd) + r(groups, 1, 1, Fd, scale=3.0)).reshape(B, N, Fd).contiguous()
    p = dict(w1=r(64, Fd, scale=0.3), b1=r(64, scale=0.2), gamma=1 + r(64, scale=0.2), beta=r(64, scale=0.3))
    eps = 1e-5
    ref, ref_stats = _grouped_ref(x, p, groups, eps)
    n_p = ops.critic_partials(B, groups)
    if groups >= 2 * L.sm_count():
        assert n_p == groups  # one slot per group
    nan = float("nan")
    stats = torch.full((groups, 2), nan, dtype=torch.float64, device="cuda")
    sp = torch.full((n_p, 2), nan, dtype=torch.float64, device="cuda")
    ysum = torch.full((B, 64), nan, device="cuda")
    d = L.GrlCriticDesc(n_graphs=B, n_tokens=N, n_feat=Fd, n_partials=n_p, eps=eps, count=float(b_env) * N * 64,
                        x=L.ptr(x), w1=L.ptr(p["w1"]), b1=L.ptr(p["b1"]), gamma=L.ptr(p["gamma"]), beta=L.ptr(p["beta"]),
                        stats=L.ptr_any(stats), stat_partials=L.ptr_any(sp), ysum=L.ptr(ysum), n_groups=groups)
    L.call("grl_critic_inner_stats", C.byref(d))
    L.call("grl_critic_inner_fwd", C.byref(d))
    assert G.rel(ysum, ref) < 1e-5, G.err_report("ysum", ysum, ref)
    assert G.rel(stats[:, 0], ref_stats[:, 0]) < 1e-5 and G.rel(stats[:, 1], ref_stats[:, 1]) < 1e-5
    # the op wraps the same launches
    out = ops.critic_inner(x, p["w1"], p["b1"], p["gamma"], p["beta"], eps, groups=groups)
    assert torch.equal(out, ysum)


def test_grouped_op_refuses_a_backward_pass():
    from geometry_rl_b200 import ops
    x = torch.randn(4, 9, 15, device="cuda")
    w1 = torch.randn(64, 15, device="cuda", requires_grad=True)
    y = ops.critic_inner(x, w1, torch.zeros(64, device="cuda"), torch.ones(64, device="cuda"), torch.zeros(64, device="cuda"),
                         1e-5, groups=2)
    with pytest.raises(AssertionError, match="grouped backward"):
        y.sum().backward()


# ---- 2. GAE.advantage against the oracle and against adv_module(td) ------------------------------------------------
def _td(roll, keys, dev=None):
    dev = dev or G.dev()
    td = {k: roll[k][:, :-1].to(dev) for k in keys}
    td["next"] = {k: roll[k][:, 1:].to(dev) for k in keys}
    td["next"].update({"reward": roll["reward"].unsqueeze(-1).to(dev), "done": roll["done"].unsqueeze(-1).to(dev),
                       "terminated": roll["terminated"].unsqueeze(-1).to(dev)})
    return td


def _copy(td):
    out = {k: v for k, v in td.items() if k != "next"}
    out["next"] = dict(td["next"])
    return out


def _outs(td):
    return [td[k] for k in OUT_KEYS] + [td["next"]["state_value"]]


@pytest.mark.parametrize("cfg_name", CONFIG_ORDER)
def test_advantage_matches_oracle(cfg_name):
    from tests.test_gpu_step import _setup
    cfg, actor, critic, loss_module, adv_module, oracle, _, gen = _setup(cfg_name)
    Benv, T = 5, 11
    roll = synthetic_rollout(cfg, gen, num_envs=Benv, rollout_len=T)
    a_ref, vt_ref, v_ref = oracle.gae(roll)
    td = adv_module.advantage(_td(roll, critic.in_keys))
    assert td["advantage"].shape == (Benv, T, 1) and td["next"]["state_value"].shape == (Benv, T, 1)
    assert G.rel(td["state_value"][..., 0], v_ref[:, :-1]) < 1e-5, G.err_report("value", td["state_value"][..., 0], v_ref[:, :-1])
    assert G.rel(td["next"]["state_value"][..., 0], v_ref[:, 1:]) < 1e-5
    assert G.rel(td["advantage"][..., 0], a_ref) < 1e-5, G.err_report("adv", td["advantage"][..., 0], a_ref)
    assert G.rel(td["value_target"][..., 0], vt_ref) < 1e-5, G.err_report("vt", td["value_target"][..., 0], vt_ref)


@pytest.mark.parametrize("cfg_name", [RIGID, CLOTH])
def test_advantage_matches_the_torch_formulation_at_a_mid_size(cfg_name):
    from geometry_rl_b200 import learner
    cfg = CONFIGS[cfg_name]
    _, critic, _, _, adv_module = learner.build_agent(cfg, G.dev(), seed=1)
    roll = synthetic_rollout(cfg, torch.Generator().manual_seed(11), num_envs=256 if cfg_name == RIGID else 64,
                             rollout_len=32)
    fused = adv_module.advantage(_td(roll, critic.in_keys))
    plain = adv_module(_td(roll, critic.in_keys))
    for k, a, b in zip(OUT_KEYS + ("next.state_value",), _outs(fused), _outs(plain)):
        assert G.rel(a, b) < 1e-5, G.err_report(k, a, b)


# ---- 3. replays: bit-identical to eager calls, between captured update and act replays --------------------------------
def test_graphed_advantage_equals_eager_between_update_and_act_replays():
    from geometry_rl_b200 import learner
    from tests.test_gpu_act import _minibatches, _obs_batches
    cfg = CONFIGS[RIGID]
    actor, critic, _, loss_module, adv_module = learner.build_agent(cfg, G.dev(), seed=2)
    Benv, T, b_update, b_act = 8, 6, 16, 8
    rolls = [_td(synthetic_rollout(cfg, torch.Generator().manual_seed(40 + i), num_envs=Benv, rollout_len=T),
                 critic.in_keys) for i in range(4)]
    mbs = _minibatches(cfg, actor, critic, b_update, 3, 500)
    obs = _obs_batches(cfg, b_act, 3, 700)
    lrn = learner.Learner(cfg, actor, critic, loss_module)
    lrn.capture(mbs[0], warmup=2)
    actor.capture_act(obs[0], seed=9)
    adv_module.capture(rolls[0])
    # an eager update at the minibatch size drops the critic builder's placeholder for Benv (T+1) graphs; the graph keeps
    # its own alive (the update changes the critic too)
    lrn.update(mbs[1])
    first = [t.clone() for t in _outs(adv_module.advantage_graphed(_copy(rolls[0])))]
    for i in range(3):
        actor.act_graphed(dict(obs[i]))
        graphed = [t.clone() for t in _outs(adv_module.advantage_graphed(_copy(rolls[i + 1])))]
        eager = _outs(adv_module.advantage(_copy(rolls[i + 1])))
        for k, a, b in zip(OUT_KEYS + ("next.state_value",), graphed, eager):
            assert torch.equal(a, b), f"replay {i}: {k} graphed != eager"
        lrn.update_graphed(mbs[i])
    # replays read the critic in place: after three updates the same rollout gives other values, equal to eager ones
    again = _outs(adv_module.advantage_graphed(_copy(rolls[0])))
    assert not torch.equal(again[2], first[2])
    for a, b in zip(again, _outs(adv_module.advantage(_copy(rolls[0])))):
        assert torch.equal(a, b)
    # advantage_static: the graph's own outputs, no copies
    out = adv_module.advantage_static()
    assert out[0].data_ptr() == adv_module.advantage_static()[0].data_ptr()
    assert torch.equal(out[0], again[0])


def test_capture_refuses_eager_rebuild_builders():
    from geometry_rl_b200 import learner
    cfg = CONFIGS[RIGID]
    _, critic, _, _, adv_module = learner.build_agent(cfg, G.dev(), seed=0)
    critic.module._network1.hyper_data.rebuild_every_call = True
    td = _td(synthetic_rollout(cfg, torch.Generator().manual_seed(1), num_envs=2, rollout_len=3), critic.in_keys)
    with pytest.raises(ValueError, match="cannot be replayed"):
        adv_module.capture(td)
    assert getattr(adv_module, "_adv_graph", None) is None


# ---- 4. two ranks, each holding half the environments ----------------------------------------------------------------
DP_CFG, DP_BENV, DP_T = RIGID, 8, 5


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_rolls(keys, dev):
    cfg = CONFIGS[DP_CFG]
    return [_td(synthetic_rollout(cfg, torch.Generator().manual_seed(60 + i), num_envs=DP_BENV, rollout_len=DP_T), keys, dev)
            for i in range(2)]


def _shard(td, sl):
    out = {k: v[sl] for k, v in td.items() if k != "next"}
    out["next"] = {k: v[sl] for k, v in td["next"].items()}
    return out


def _dp_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from geometry_rl_b200 import learner
        from geometry_rl_b200.parallel import DataParallel
        dev = torch.device("cuda", rank if torch.cuda.device_count() >= world else 0)
        torch.cuda.set_device(dev)
        _, critic, _, loss_module, adv_module = learner.build_agent(CONFIGS[DP_CFG], dev, seed=0)
        DataParallel().attach(loss_module)
        sl = slice(rank * DP_BENV // world, (rank + 1) * DP_BENV // world)
        rolls = [_shard(td, sl) for td in _dp_rolls(critic.in_keys, dev)]
        eager = [[t.cpu() for t in _outs(adv_module.advantage(_copy(td)))] for td in rolls]
        adv_module.capture(rolls[0])
        graphed = [[t.cpu() for t in _outs(adv_module.advantage_graphed(_copy(td)))] for td in rolls]
        torch.cuda.synchronize()
        torch.save({"eager": eager, "graphed": graphed}, os.path.join(out_dir, f"rank{rank}.pt"))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_ranks_give_the_single_process_advantages(tmp_path):
    from geometry_rl_b200 import learner
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, str(tmp_path))) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    res = [torch.load(tmp_path / f"rank{r}.pt", weights_only=True) for r in range(world)]
    _, critic, _, _, adv_module = learner.build_agent(CONFIGS[DP_CFG], G.dev(), seed=0)
    for i, td in enumerate(_dp_rolls(critic.in_keys, G.dev())):
        single = _outs(adv_module.advantage(_copy(td)))
        for mode in ("eager", "graphed"):
            for j, name in enumerate(OUT_KEYS + ("next.state_value",)):
                got = torch.cat([res[r][mode][i][j] for r in range(world)], 0)
                assert G.rel(got, single[j]) < 1e-6, f"rollout {i} {mode}: " + G.err_report(name, got, single[j])
