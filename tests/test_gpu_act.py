"""GPU: the rollout-time acting path (grl_gaussian_act + grl_act_advance, PolicyOperator.act / capture_act /
act_graphed).  The kernel against an fp64 torch evaluation of the head on random heads and against the numpy Philox
reference (tests/philox_reference.py); the noise's statistics at a fixed seed; determinism; the five configs through
the public interface, eager and replayed; acting graphs interleaved with captured updates; the capture guard."""
import dataclasses
import math

import numpy as np
import pytest
import torch

from geometry_rl_b200.synthetic import CONFIGS, CONFIG_ORDER, synthetic_minibatch, synthetic_obs
from tests import gpu_helpers as G
from tests import philox_reference as P

pytestmark = pytest.mark.gpu

LOG_2PI = math.log(2.0 * math.pi)
SHIFT = float(torch.log(torch.expm1(torch.tensor(1.0 - 1e-5))))  # GNNGaussianPolicyDiag._pre_activation_shift
MIN_STD = float(torch.tensor(1e-5))
ROPE, RIGID, CLOTH = "rope_shaping_hepi_trpl_cfg", "rigid_insertion_multi_hepi_trpl_cfg", "cloth_hanging_multi_hepi_trpl_cfg"
SIZES = {RIGID: 16, "rigid_pushing_multi_empn_trpl_cfg": 16, CLOTH: 8, ROPE: 6,
         "rigid_insertion_two_agents_multi_transformer_trpl_cfg": 12}


@pytest.fixture
def sixteen_bit():
    from geometry_rl_b200 import ops
    ops.set_precision("bf16")
    yield
    ops.set_precision("fp32")


def _state(seed, call):
    return torch.tensor([seed, call], dtype=torch.int64, device=G.dev())


def _head(B, A, a, post_fc, contextual, gen):
    """Random head inputs: pre-activations spread over [-30, 30] (both sides of torch's Softplus threshold 20)."""
    k = A * a
    h = torch.randn(B * A, 64, generator=gen)
    p = {"hidden": h if (post_fc or contextual) else None,
         "mean": None if post_fc else torch.randn(B, k, generator=gen) * 0.7,
         "mean_weight": torch.randn(a, 64, generator=gen) * 0.2 if post_fc else None,
         "mean_bias": torch.randn(a, generator=gen) * 0.1 if post_fc else None}
    if contextual:
        p["std_weight"] = torch.randn(a, 64, generator=gen) * 0.05
        p["std_bias"] = torch.linspace(-30.0, 30.0, a)
    else:
        p["std_weight"], p["std_bias"] = torch.linspace(-30.0, 30.0, a), None
    return p


def _head_fp64(p, B, A, a, tanh_mean):
    d = {k: (v.double() if v is not None else None) for k, v in p.items()}
    if d["mean"] is None:
        mean = (d["hidden"] @ d["mean_weight"].T + d["mean_bias"]).reshape(B, A * a)
        if tanh_mean:
            mean = torch.tanh(mean)
    else:
        mean = d["mean"].reshape(B, A * a)
    pre = d["hidden"] @ d["std_weight"].T + d["std_bias"] if d["std_bias"] is not None else d["std_weight"].expand(B * A, a)
    x = pre + SHIFT
    sd = (torch.where(x > 20.0, x, torch.log1p(torch.exp(x))) + MIN_STD).reshape(B, A * a)
    return mean, sd


@pytest.mark.parametrize("A,a", [(1, 3), (2, 3), (4, 3), (4, 8)])
@pytest.mark.parametrize("post_fc", [False, True])
@pytest.mark.parametrize("contextual", [False, True])
def test_kernel_matches_fp64_head_and_philox_reference(A, a, post_fc, contextual):
    from geometry_rl_b200 import ops
    B, k = 37, A * a
    gen = torch.Generator().manual_seed(100 * A + 10 * a + 2 * post_fc + contextual)
    p = _head(B, A, a, post_fc, contextual, gen)
    tanh_mean = post_fc and contextual
    seed, call = 0x5EED00000001 + k, 3
    dp = {kk: (v.to(G.dev()) if v is not None else None) for kk, v in p.items()}
    loc, cov, action, logp, eps = ops.gaussian_act(_state(seed, call), batch=B, num_rows=A, action_dim=a,
                                                   pre_shift=SHIFT, minimal_std=MIN_STD, use_tanh_mean=tanh_mean,
                                                   return_eps=True, **dp)
    mean64, sd64 = _head_fp64(p, B, A, a, tanh_mean)
    var64 = sd64 * sd64
    loc, cov, action, logp, eps = (t.cpu() for t in (loc, cov, action, logp, eps))
    assert loc.shape == (B, k) and cov.shape == (B, k, k) and logp.shape == (B,)
    var = torch.diagonal(cov, dim1=-2, dim2=-1)
    assert bool(((loc.double() - mean64).abs() <= 1e-6 * mean64.abs()).all()), G.err_report("loc", loc, mean64)
    assert bool(((var.double() - var64).abs() <= 1e-6 * var64).all()), G.err_report("var", var, var64)
    assert bool((cov * (1 - torch.eye(k))).eq(0).all()) and int((cov != 0).sum()) == B * k  # exact zeros off the diagonal
    ref_eps = torch.from_numpy(P.act_eps(seed, call, B, k))
    assert float((eps - ref_eps).abs().max()) <= 1e-5
    act_ref = loc.double() + eps.double() * sd64
    assert bool(((action.double() - act_ref).abs() <= 1e-6 * (loc.double().abs() + (eps.double() * sd64).abs())).all())
    lp_ref = -0.5 * (((action.double() - loc.double()) ** 2 / var.double()).sum(-1) + k * LOG_2PI
                     + var.double().log().sum(-1))
    assert bool(((logp.double() - lp_ref).abs() <= 1e-6 * lp_ref.abs()).all()), G.err_report("log_prob", logp, lp_ref)
    # evaluation mode: action = loc, nothing drawn
    loc_d, _, act_d, lp_d, eps_d = ops.gaussian_act(_state(seed, call), batch=B, num_rows=A, action_dim=a,
                                                    pre_shift=SHIFT, minimal_std=MIN_STD, use_tanh_mean=tanh_mean,
                                                    deterministic=True, return_eps=True, **dp)
    assert torch.equal(act_d, loc_d) and torch.equal(loc_d.cpu(), loc) and not bool(eps_d.any())
    lp_d_ref = -0.5 * (k * LOG_2PI + var.double().log().sum(-1))
    assert bool(((lp_d.cpu().double() - lp_d_ref).abs() <= 1e-6 * lp_d_ref.abs()).all())


def _draw(B, k, seed, call, rank=0):
    from geometry_rl_b200 import ops
    A, a = (1, k)
    p = {"std_weight": torch.zeros(a, device=G.dev()), "mean": torch.zeros(B, k, device=G.dev())}
    return ops.gaussian_act(_state(seed, call), batch=B, num_rows=A, action_dim=a, pre_shift=SHIFT, minimal_std=MIN_STD,
                            rank=rank, return_eps=True, **p)[4]


def test_noise_statistics_at_a_fixed_seed():
    """KS test of 2^20 draws against N(0, 1); correlations between the 8 components over 2^20 samples and between the
    draws of two consecutive calls below 5e-3 (a fixed seed: the outcome is deterministic)."""
    from scipy import stats
    B, k, seed = 1 << 20, 8, 20261021
    z0 = _draw(B, k, seed, 0).double().cpu().numpy()
    z1 = _draw(B, k, seed, 1).double().cpu().numpy()
    assert stats.kstest(z0.reshape(-1)[: 1 << 20], "norm").pvalue > 1e-3
    c = np.corrcoef(z0, rowvar=False)
    assert float(np.abs(c - np.eye(k)).max()) < 5e-3
    assert abs(float(np.corrcoef(z0.reshape(-1), z1.reshape(-1))[0, 1])) < 5e-3
    assert abs(z0.mean()) < 5e-3 and abs(z0.std() - 1.0) < 5e-3


def test_draws_are_deterministic_and_independent_of_the_grid():
    from geometry_rl_b200 import _lib
    B, k, seed = 20000, 12, 77  # more samples than one grid-stride pass covers
    ref = _draw(B, k, seed, 5)
    assert torch.equal(_draw(B, k, seed, 5), ref)
    _lib.reserve_sms(4)
    try:
        assert torch.equal(_draw(B, k, seed, 5), ref)
    finally:
        _lib.reserve_sms(0)
    assert torch.equal(_draw(100, k, seed, 5), ref[:100])  # nor on the batch size
    for other in (_draw(B, k, seed, 6), _draw(B, k, seed + 1, 5), _draw(B, k, seed, 5, rank=1)):
        assert float((other != ref).float().mean()) > 0.99
    ranked = _draw(64, k, seed, 5, rank=2).cpu()
    assert float((ranked - torch.from_numpy(P.act_eps(seed, 5, 64, k, rank=2))).abs().max()) <= 1e-5
    # grl_act_advance: one increment per launch
    from geometry_rl_b200 import ops
    st = _state(seed, 41)
    ops.act_advance(st)
    ops.act_advance(st)
    assert st.tolist() == [seed, 43]


def _agent(cfg_name, seed=0):
    from geometry_rl_b200 import learner
    cfg = CONFIGS[cfg_name]
    actor, critic, _, loss_module, _ = learner.build_agent(cfg, G.dev(), seed=seed)
    return cfg, actor, critic, loss_module


def _obs_batches(cfg, B, n, seed):
    """`n` observation batches of the same B environments (same geometries per slot), other states."""
    from geometry_rl_b200.tensors import to_device
    env_ids = torch.arange(B) * max(1, cfg.num_envs // B) % cfg.num_envs
    return [to_device(synthetic_obs(cfg, B, torch.Generator().manual_seed(seed + i), env_ids=env_ids), G.dev())
            for i in range(n)]


def _outs(td):
    return [td[k].clone() for k in ("loc", "covariance_matrix", "action", "sample_log_prob")]


@pytest.mark.parametrize("cfg_name", CONFIG_ORDER)
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_configs_graphed_equals_eager_and_matches_get_dist(cfg_name, precision):
    from geometry_rl_b200 import ops
    from geometry_rl_b200.algorithms.trust_region_projections.objectives.operators import DiagMultivariateNormal
    ops.set_precision(precision)
    try:
        cfg, actor, _, _ = _agent(cfg_name)
        B = SIZES[cfg_name]
        obs = _obs_batches(cfg, B, 4, 300)
        with torch.no_grad():
            actor.get_dist(obs[0])  # calibration + topology from the first batch, as capture_act does
        actor.set_act_state(1234, 0)
        eager = []
        for td in obs[1:]:
            td = dict(td)
            actor.act(td)
            eager.append(_outs(td))
            dist = actor.get_dist(td)
            assert G.rel(td["loc"], dist.mean) <= 1e-6, G.err_report("loc", td["loc"], dist.mean)
            var = torch.diagonal(td["covariance_matrix"], dim1=-2, dim2=-1)
            assert G.rel(var, dist.var_diag) <= 1e-6, G.err_report("var", var, dist.var_diag)
            lp = DiagMultivariateNormal(td["loc"], var_diag=var).log_prob(td["action"])
            assert G.rel(td["sample_log_prob"], lp) <= 1e-5, G.err_report("log_prob", td["sample_log_prob"], lp)
            assert not torch.equal(td["action"], td["loc"])
        assert actor.act_state() == (1234, 3)
        actor.capture_act(obs[0], seed=1234)
        for td, ref in zip(obs[1:], eager):
            td = dict(td)
            actor.act_graphed(td)
            for got, exp, name in zip(_outs(td), ref, ("loc", "covariance_matrix", "action", "sample_log_prob")):
                assert torch.equal(got, exp), f"{name}: graphed != eager"
        assert actor.act_state() == (1234, 3)
        # act_static: zero-copy outputs of the replay on the static inputs
        out = actor.act_static()
        assert out["action"].data_ptr() == actor.act_static()["action"].data_ptr()
        # evaluation: action = loc, and the stream does not move
        td = dict(obs[1])
        actor.act(td, deterministic=True)
        assert torch.equal(td["action"], td["loc"]) and torch.equal(td["loc"], eager[0][0])
        assert actor.act_state() == (1234, 5)
    finally:
        ops.set_precision("fp32")


def _minibatches(cfg, actor, critic, B, n, seed):
    """Update minibatches around the freshly initialised head (mean 0, var 1, value 0), like bench.py's inputs."""
    from geometry_rl_b200.tensors import to_device
    gen = torch.Generator().manual_seed(seed)
    k = cfg.total_action_dim
    out = []
    for i in range(n):
        env_ids = torch.arange(B) * max(1, cfg.num_envs // B) % cfg.num_envs
        obs = synthetic_obs(cfg, B, torch.Generator().manual_seed(seed + 100 + i), env_ids=env_ids)
        mb = synthetic_minibatch(obs, torch.zeros(B, k), torch.ones(B, k), torch.zeros(B, 1), gen)
        out.append(to_device(mb, G.dev()))
    return out


@pytest.mark.parametrize("cfg_name,b_act,b_update", [(RIGID, 16, 16), (CLOTH, 8, 16)])
def test_act_replays_between_update_replays_leave_the_update_unchanged(cfg_name, b_act, b_update):
    from geometry_rl_b200 import learner
    finals = {}
    for with_act in (False, True):
        cfg, actor, critic, loss_module = _agent(cfg_name, seed=2)
        cfg = dataclasses.replace(cfg, clip_grad_norm=False)
        mbs = _minibatches(cfg, actor, critic, b_update, 3, 500)
        obs = _obs_batches(cfg, b_act, 3, 700)
        lrn = learner.Learner(cfg, actor, critic, loss_module)
        lrn.capture(mbs[0], warmup=2)
        if with_act:
            actor.capture_act(obs[0], seed=9)
        for i in range(3):
            if with_act:
                actor.act_graphed(dict(obs[i]))
            lrn.update_graphed(mbs[i])
        torch.cuda.synchronize()
        finals[with_act] = torch.cat([p.detach().reshape(-1).clone() for p in list(actor.parameters()) + list(critic.parameters())])
        if with_act:  # the act graph reads the parameters in place: a replay now equals an eager act on the updated weights
            state = actor.act_state()
            replayed, eager = dict(obs[0]), dict(obs[0])
            actor.act_graphed(replayed)
            actor.set_act_state(*state)
            actor.act(eager)
            for got, exp in zip(_outs(replayed), _outs(eager)):
                assert torch.equal(got, exp)
    assert torch.equal(finals[True], finals[False])


def test_radius_refresh_act_replays_follow_the_positions(sixteen_bit):
    from tests.test_gpu_radius import RADIUS
    cfg, actor, _, _ = _agent(ROPE, seed=4)
    hd = actor.policy.hyper_data
    hd.internal_edges = "radius"
    hd.radius, hd.max_num_neighbors = RADIUS[ROPE]
    hd.rebuild_every_call = True
    assert hd.refresh_in_place()
    obs = _obs_batches(cfg, 6, 4, 900)  # the rope moves from batch to batch
    actor.capture_act(obs[0], seed=31)
    graphed = []
    for td in obs[1:]:
        td = dict(td)
        actor.act_graphed(td)
        graphed.append(_outs(td))
    actor.set_act_state(31, 0)
    for td, ref in zip(obs[1:], graphed):
        td = dict(td)
        actor.act(td)
        for got, exp in zip(_outs(td), ref):
            assert torch.equal(got, exp)
    assert not torch.equal(graphed[0][0], graphed[1][0])


def test_capture_act_refuses_eager_rebuild_modes():
    from geometry_rl_b200 import ops
    for internal, precision in (("knn", "bf16"), ("radius", "fp32")):
        ops.set_precision(precision)
        try:
            cfg, actor, _, _ = _agent(ROPE)
            hd = actor.policy.hyper_data
            if internal == "radius":
                hd.internal_edges, hd.radius, hd.max_num_neighbors = "radius", 0.025, 8
            hd.rebuild_every_call = True
            obs = _obs_batches(cfg, 4, 1, 5)[0]
            with pytest.raises(ValueError, match="cannot be replayed"):
                actor.capture_act(obs, seed=0)
            assert getattr(actor, "_act_graph", None) is None and getattr(actor, "_act_static", None) is None
        finally:
            ops.set_precision("fp32")
