"""GPU: TRPL entropy control on the fused loss path (grl_trpl_entropy_bound, the entropy fields of grl_trpl_fwd / _bwd).

1. the projection kernels alone against an fp64 autograd restatement (oracle KL / W2 projections + the entropy
   projections), {KL, W2} x {inequality, equality} x {after, first}, k of the configs, masks mixed;
2. the bound and the latched initial entropy against the fp64 restatement, both schedules, several steps;
3. fused against unfused TRPLLoss with entropy control on all five configs;
4. Learner.fit graphed against eager, bit for bit, with a moving bound: first latch, re-capture, set_step resume;
5. two gloo ranks sharing one GPU against the single process."""
import ctypes as C
import math
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from geometry_rl_b200.synthetic import CONFIGS, synthetic_minibatch, synthetic_obs
from tests import entropy_reference as R
from tests import gpu_helpers as G

pytestmark = pytest.mark.gpu

SIZES = {"rigid_insertion_multi_hepi_trpl_cfg": 48, "rigid_pushing_multi_empn_trpl_cfg": 40,
         "cloth_hanging_multi_hepi_trpl_cfg": 24, "rope_shaping_hepi_trpl_cfg": 6,
         "rigid_insertion_two_agents_multi_transformer_trpl_cfg": 16}
KEYS = ("loss_objective", "loss_trust_region", "loss_entropy", "loss_critic", "ESS", "kl", "constraint", "mean_constraint",
        "mean_constraint_max", "cov_constraint", "cov_constraint_max", "entropy", "entropy_diff")


# ---- 1. the projection kernels alone ---------------------------------------------------------------------------------
@pytest.mark.parametrize("k", sorted({c.total_action_dim for c in CONFIGS.values()}))
@pytest.mark.parametrize("first", [False, True], ids=["after", "first"])
@pytest.mark.parametrize("equality", [False, True], ids=["ineq", "eq"])
@pytest.mark.parametrize("proj_type", ["kl", "w2"])
def test_projection_kernels_match_fp64(proj_type, equality, first, k):
    from geometry_rl_b200 import _lib as L
    gen = torch.Generator().manual_seed(1000 + 10 * k + 2 * first + equality)
    B0, em, ec = 600, 0.05, 0.0025
    q_mean = torch.randn(B0, k, generator=gen) * 0.3
    q_v = (0.5 + torch.rand(B0, k, generator=gen)) ** 2
    s = torch.rand(B0, 1, generator=gen)
    mean = q_mean + torch.randn(B0, k, generator=gen) * 0.5 * s
    v = q_v * torch.exp(torch.randn(B0, k, generator=gen) * 0.3 * s)
    D = torch.float64
    # the bound sits at the median of the entropies the entropy projection sees; samples within 1e-4 of it are dropped
    with torch.no_grad():
        x = v.to(D) if first else R.project(mean.to(D), v.to(D), q_mean.to(D), q_v.to(D), em, ec, proj_type, -math.inf,
                                            False, False)[1]
        h = R.entropy(x)
        beta = float(h.median())
        keep = (h - beta).abs() > 1e-4
    q_mean, q_v, mean, v = (t[keep].contiguous().cuda() for t in (q_mean, q_v, mean, v))
    B = mean.shape[0]
    g_pm, g_pv, am, av = (torch.randn(B, k, generator=gen).cuda() for _ in range(4))

    nan = lambda *s_, dt=torch.float32: torch.full(s_, float("nan"), dtype=dt, device="cuda")
    beta_t = torch.tensor([beta], dtype=D, device="cuda")
    pm, pv, alpha, eta = nan(B, k), nan(B, k), nan(B, dt=D), nan(B, 2, dt=D)
    mode = L.ENTROPY_MODE["eq" if equality else "ineq"]
    d = L.GrlProjDesc(batch=B, k=k, proj_type={"kl": 0, "w2": 1}[proj_type], eps_mean=em, eps_cov=ec, mean=L.ptr(mean),
                      v=L.ptr(v), old_mean=L.ptr(q_mean), old_v=L.ptr(q_v), proj_mean=L.ptr(pm), proj_v=L.ptr(pv),
                      eta=L.ptr(eta), entropy_mode=mode, entropy_first=int(first), entropy_beta=L.ptr(beta_t),
                      entropy_alpha=L.ptr(alpha))
    L.call("grl_trpl_fwd", C.byref(d))
    gm, gv = nan(B, k), nan(B, k)
    d.grad_proj_mean, d.grad_proj_v, d.grad_mean, d.grad_v = L.ptr(g_pm), L.ptr(g_pv), L.ptr(gm), L.ptr(gv)
    d.grad_mean_add, d.grad_v_add, d.entropy_beta = L.ptr(am), L.ptr(av), None  # the backward reads alpha only
    L.call("grl_trpl_bwd", C.byref(d))
    torch.cuda.synchronize()

    m64, v64 = mean.to(D).requires_grad_(True), v.to(D).requires_grad_(True)
    rpm, rpv = R.project(m64, v64, q_mean.to(D), q_v.to(D), em, ec, proj_type, beta, equality, first)
    ((g_pm.to(D) * rpm).sum() + (g_pv.to(D) * rpv).sum() + (am.to(D) * m64).sum() + (av.to(D) * v64).sum()).backward()
    # W2: the trust-region weight comes from the fp32 sum of 1 + (v/vo)^2 - 2 v/vo, as in the reference; its rounding
    # puts the fp32 W2 covariance gradient 2e-5 .. 5e-5 from fp64 whatever the entropy control does
    # (test_oracle_golden.py::test_w2_grad_noise_floor), the 1e-4 bound of the other GPU tests
    gtol = 1e-4 if proj_type == "w2" else 1e-5
    bad = [G.err_report(n, a, b) for n, a, b, tol in (("proj_mean", pm, rpm, 1e-5), ("proj_v", pv, rpv, 1e-5),
                                                      ("grad_mean", gm, m64.grad, 1e-5), ("grad_v", gv, v64.grad, gtol))
           if not G.rel(a, b) < tol]
    assert not bad, "\n".join(bad)
    active = alpha != 1.0
    assert bool(active.all()) if equality else 0.2 < float(active.double().mean()) < 0.8, "the mask is not mixed"


# ---- 2. the bound ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["linear", "exp"])
def test_bound_and_initial_entropy_match_the_restatement(kind):
    from geometry_rl_b200 import ops
    gen = torch.Generator().manual_seed(5)
    k, T, te, temp = 6, 50, -0.7, 0.6
    state = torch.zeros(4, dtype=torch.float64, device="cuda")
    step = torch.zeros((), dtype=torch.int64, device="cuda")
    ent = ops.EntropyControl(state, step, kind, T, te, temp, False, False)
    first_v = None
    for i, s in enumerate((0, 1, 3, 17, 50, 80)):
        old_v = ((0.3 + torch.rand(4096 + 37 * i, k, generator=gen)) ** 2).cuda()
        first_v = old_v if first_v is None else first_v
        step.fill_(s)
        assert ops.entropy_bound(ent, old_v) == 1
        ie_ref = float(R.entropy(first_v.double()).mean())  # latched on the first call only
        ie, flag, b = (float(x) for x in state[:3].cpu())
        assert flag == 1.0 and abs(ie - ie_ref) <= 1e-12 * abs(ie_ref), (ie, ie_ref)
        assert abs(b - float(R.schedule(kind, ie, te, temp, s, T, k))) <= 1e-14 * max(1.0, abs(b)), s
        assert abs(b - float(R.schedule(kind, ie_ref, te, temp, s, T, k))) <= 1e-11 * max(1.0, abs(b))


# ---- 3. fused against unfused TRPLLoss ----------------------------------------------------------------------------------
def _agent(cfg_name, B, proj_type="kl", seed=0, dev=None, in_place=False, **pkw):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    dev = dev or G.dev()
    cfg = CONFIGS[cfg_name]
    actor, critic, projection, loss_module, _ = learner.build_agent(cfg, dev, proj_type=proj_type, seed=seed,
                                                                    projection_kwargs=pkw)
    if in_place:  # the kNN topology of every minibatch is rebuilt on the device, inside the replay too
        hd = actor.get_submodule("0").module.hyper_data
        hd.rebuild_every_call, hd.knn_in_place = True, True
    gen = torch.Generator().manual_seed(31 + seed)
    obs = synthetic_obs(cfg, B, gen, env_ids=torch.arange(B) * max(1, cfg.num_envs // B) % cfg.num_envs)
    with torch.no_grad():  # calibration before the minibatch is drawn from the policy
        d = actor.get_dist(to_device(obs, dev))
        v = critic.module(*[obs[k_].to(dev) for k_ in critic.in_keys])
    mb = synthetic_minibatch(obs, d.mean, d.var_diag, v, gen)
    return cfg, actor, critic, projection, loss_module, mb


def _target_for(kind, ie, beta, step, T, k, temp):
    """target_entropy that puts the bound at `beta` on `step` (so the inequality mask is partly active)."""
    if kind == "linear":
        return ie + (beta - ie) * T / step
    r = temp ** (10 * step / T)
    return (beta - ie * r) / (k * (1 - r))


def _old_entropy(mb):
    return float(R.entropy(torch.diagonal(mb["covariance_matrix"], dim1=-2, dim2=-1).double()).mean())


MODES = [("linear", False, False, "kl"), ("exp", True, True, "kl"), ("linear", False, True, "kl"),
         ("exp", True, False, "kl"), ("linear", False, True, "w2")]


@pytest.mark.parametrize("mode", MODES, ids=["-".join(str(x) for x in m) for m in MODES])
@pytest.mark.parametrize("cfg_name", list(SIZES))
def test_fused_and_unfused_loss_modules_agree_with_entropy_control(cfg_name, mode):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    kind, eq, first, proj_type = mode
    if (mode != MODES[0] and mode != MODES[1]) and cfg_name != "rigid_insertion_multi_hepi_trpl_cfg":
        pytest.skip("every mode on one config, two modes on all five")
    T, step, temp = 20, 3, 0.6
    cfg, actor, critic, pr, loss_module, mb = _agent(cfg_name, SIZES[cfg_name], proj_type, entropy_schedule=kind,
                                                     entropy_eq=eq, entropy_first=first, total_train_steps=T,
                                                     temperature=temp)
    ie = _old_entropy(mb)
    pr.target_entropy = torch.tensor(_target_for(kind, ie, ie - 0.02, step, T, cfg.total_action_dim, temp))
    lrn = learner.Learner(cfg, actor, critic, loss_module)
    lrn.set_step(step)
    res = {}
    for fused in (True, False):
        loss_module.fused = fused
        actor.zero_grad(set_to_none=True)
        out = lrn.compute_losses(to_device(mb, G.dev()))
        out["actor_loss"].backward()
        res[fused] = ({k_: float(t) for k_, t in out.items()},
                      {k_: p.grad.detach().clone() for k_, p in actor.named_parameters() if p.grad is not None})
    (o1, g1), (o0, g0) = res[True], res[False]
    assert set(o1) == set(o0) and set(g1) == set(g0)
    # entropy_diff: the torch formulation subtracts two fp32 entropies of about 10, whose spacing is 1e-6
    bad = [f"{k_}: {o1[k_]} vs {o0[k_]}" for k_ in o0
           if not abs(o1[k_] - o0[k_]) <= 1e-5 * abs(o0[k_]) + (2e-6 if k_ == "entropy_diff" else 2e-7)]
    # the torch formulation differentiates the entropy projection in fp32, where the two terms of
    # alpha g_j - alpha / (k v_j) sum_i g_i v_i cancel: measured up to 1.3e-5 on the smallest bias gradients
    bad += [G.err_report(k_, g1[k_], g0[k_]) for k_ in g0 if G.rel(g1[k_], g0[k_]) >= 2e-5]
    assert not bad, "\n".join(bad)
    # the device state: initial entropy of the minibatch, the bound the torch schedule gives at this step
    assert abs(float(pr.initial_entropy) - ie) <= 1e-6 * abs(ie)
    assert abs(float(pr.entropy_bound) - float(pr.get_entropy_bound(step))) <= 1e-6 * max(1.0, abs(ie))
    assert abs(float(pr.entropy_bound) - (ie - 0.02)) < 1e-4


def test_two_stream_update_advances_the_device_step_and_capture_refuses_the_torch_path():
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    cfg, actor, critic, pr, loss_module, mb = _agent("rope_shaping_hepi_trpl_cfg", 6, entropy_schedule="linear")
    lrn = learner.Learner(cfg, actor, critic, loss_module)
    assert lrn._critic_stream is not None and loss_module.step_counter is lrn._step
    batch = to_device(mb, G.dev())
    for _ in range(2):
        lrn.update(batch)
    lrn.capture(batch)
    lrn.update_graphed(batch)
    torch.cuda.synchronize()
    assert int(lrn._step) == lrn.num_network_updates == 3
    # a direct call outside the learner writes the host step into the counter
    loss_module.steps_on_device, loss_module._global_steps = False, 11
    loss_module(batch)
    assert int(loss_module.step_counter) == 11
    assert float(pr.entropy_bound) == float(R.schedule("linear", float(pr.initial_entropy), 0.0, 0.5, 11, 1000, 6))
    loss_module.steps_on_device, loss_module.fused = True, False
    with pytest.raises(NotImplementedError, match="entropy schedule"):
        lrn.capture(batch)


# ---- 4. graphed equals eager ------------------------------------------------------------------------------------------
FIT_CFG, FIT_FRAMES, FIT_MB, FIT_T = "rigid_pushing_multi_empn_trpl_cfg", 96, 32, 20


@pytest.fixture
def sixteen_bit():
    from geometry_rl_b200 import ops
    ops.set_precision("bf16")
    yield
    ops.set_precision("fp32")


def _fit_run(graphed):
    """EMPN on the 16-bit path with the in-place kNN rebuild: every minibatch gets its own topology in both modes, so the
    replay and the eager update compute the same thing (as in test_gpu_empn_refresh.py's fit test)."""
    import dataclasses
    from geometry_rl_b200 import learner
    from geometry_rl_b200.rollout import DeviceRolloutBuffer
    from geometry_rl_b200.tensors import to_device
    torch.manual_seed(0)
    cfg, actor, critic, pr, loss_module, mb = _agent(FIT_CFG, FIT_FRAMES, seed=3, in_place=True,
                                                     entropy_schedule="linear", total_train_steps=FIT_T)
    cfg = dataclasses.replace(cfg, clip_grad_norm=False)
    ie = _old_entropy(mb)
    pr.target_entropy = torch.tensor(ie - 0.01 * FIT_T)  # the bound starts at ie and falls by 0.01 per update
    frames = {k_: v for k_, v in to_device(mb, G.dev()).items() if torch.is_tensor(v)}
    buf = DeviceRolloutBuffer(FIT_FRAMES, FIT_MB, G.dev(), drop_last=True, generator=torch.Generator().manual_seed(7))
    buf.extend(frames)
    lrn = learner.Learner(cfg, actor, critic, loss_module, overlap_critic=False)
    snaps = []

    def snap(res):
        torch.cuda.synchronize()
        snaps.append({"params": torch.cat([p.detach().reshape(-1).clone() for p in list(actor.parameters())
                                           + list(critic.parameters())]),
                      "losses": torch.stack([res[-1][k_].detach().reshape(()) for k_ in KEYS]).clone(),
                      "state": pr.entropy_state(G.dev()).clone(), "step": lrn._step.clone(),
                      "n": lrn.num_network_updates})

    snap(lrn.fit(buf, epochs=2, graphed=graphed))
    if graphed:  # re-capture after updates: restores what its warm-up moved
        lrn.capture({k_: v[:FIT_MB] for k_, v in frames.items()})
    snap(lrn.fit(buf, epochs=1, graphed=graphed))
    lrn.set_step(2)  # resume at another step: the bound follows the device counter
    snap(lrn.fit(buf, epochs=1, graphed=graphed))
    return snaps, frames


def test_fit_graphed_equals_eager_with_a_moving_bound(sixteen_bit):
    from geometry_rl_b200.rollout import DeviceRolloutBuffer
    eager, frames = _fit_run(False)
    graphed, _ = _fit_run(True)
    for i, (a, b) in enumerate(zip(graphed, eager)):
        for key in ("params", "losses", "state", "step"):
            assert torch.equal(a[key], b[key]), f"phase {i}: {key} graphed != eager"
        assert a["n"] == b["n"] == int(a["step"])
    assert [s["n"] for s in eager] == [6, 9, 5]
    # the initial entropy comes from the first permuted minibatch, not from the capture example
    buf = DeviceRolloutBuffer(FIT_FRAMES, FIT_MB, G.dev(), drop_last=True, generator=torch.Generator().manual_seed(7))
    buf.extend(frames)
    first = buf.sample_indices()[0]
    var = torch.diagonal(frames["covariance_matrix"], dim1=-2, dim2=-1).double()
    ie_first, ie_head = float(R.entropy(var[first]).mean()), float(R.entropy(var[:FIT_MB]).mean())
    ie = float(graphed[0]["state"][0])
    assert abs(ie - ie_first) <= 1e-12 * abs(ie_first) and abs(ie - ie_head) > 1e-9
    bound = [float(s["state"][2]) for s in eager]  # the bound of the last update of each phase
    assert bound[0] > bound[1] and bound[2] > bound[0]


# ---- 5. data parallelism -----------------------------------------------------------------------------------------------
DP_CFG, DP_B, DP_UPDATES = "rigid_insertion_multi_hepi_trpl_cfg", 16, 3


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_run(dev, shard=None, dp=None):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.tensors import to_device
    cfg, actor, critic, pr, loss_module, mb = _agent(DP_CFG, DP_B, dev=dev, entropy_schedule="exp", entropy_eq=False,
                                                     total_train_steps=10, temperature=0.5)
    ie = _old_entropy(mb)
    pr.target_entropy = torch.tensor(_target_for("exp", ie, ie - 0.02, 1, 10, cfg.total_action_dim, 0.5))
    batch = {k_: (v[shard] if torch.is_tensor(v) and shard is not None else v) for k_, v in mb.items()}
    lrn = learner.Learner(cfg, actor, critic, loss_module, dp=dp)
    for _ in range(DP_UPDATES):
        lrn.update(to_device(batch, dev))
    torch.cuda.synchronize()
    return {"params": torch.cat([p.detach().reshape(-1) for p in actor.parameters()]).cpu(),
            "state": pr.entropy_state(dev).cpu(), "step": lrn._step.cpu()}


def _dp_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from geometry_rl_b200.parallel import DataParallel
        dev = torch.device("cuda", rank if torch.cuda.device_count() >= world else 0)
        torch.cuda.set_device(dev)
        res = _dp_run(dev, slice(rank * DP_B // world, (rank + 1) * DP_B // world), DataParallel())
        torch.save(res, os.path.join(out_dir, f"rank{rank}.pt"))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_ranks_share_the_bound_and_match_the_single_process(tmp_path):
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, str(tmp_path))) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    res = [torch.load(tmp_path / f"rank{r}.pt", weights_only=True) for r in range(world)]
    assert torch.equal(res[0]["state"], res[1]["state"]), "ranks hold different entropy bounds"
    assert torch.equal(res[0]["params"], res[1]["params"])
    single = _dp_run(G.dev())
    assert int(res[0]["step"]) == int(single["step"]) == DP_UPDATES
    for i in (0, 2):  # initial entropy, bound: the global mean, equal to the single process up to summation order
        a, b = float(res[0]["state"][i]), float(single["state"][i])
        assert abs(a - b) <= 1e-6 * abs(b), (i, a, b)
    assert G.rel(res[0]["params"], single["params"]) < 1e-6, G.err_report("params", res[0]["params"], single["params"])
