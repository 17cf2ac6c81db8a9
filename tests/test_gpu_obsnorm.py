"""GPU: observation normalisation on the device (NDVecNorm.apply_device, csrc/grl_obsnorm.cu) and the acting graph that
starts from the raw observations (PolicyOperator.capture_act(obs_norm=...)).

1. the kernels against torch `__call__` on CUDA (same state: bit for bit) and against the fp64 running statistics of
   tests/test_transforms.py over ten steps, at M = 1, a ragged last CTA and every config's num_envs;
2. bit-identical results under grl_reserve_sms(0) and (4);
3. graphed equals eager for all five configs, capture leaves the statistics alone, frozen captures, restored state;
4. two ranks (gloo, one GPU) each normalising half of the environments."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from geometry_rl_b200.synthetic import CONFIGS, CONFIG_ORDER, synthetic_obs
from geometry_rl_b200.torchrl.envs import NDVecNorm
from tests import gpu_helpers as G
from tests.test_transforms import _naive

pytestmark = pytest.mark.gpu

IN_KEYS = ["position_vectors", "velocity_vectors"]
OUT_KEYS = ["norm_position_vectors", "norm_velocity_vectors"]
ACT_KEYS = ("loc", "covariance_matrix", "action", "sample_log_prob")


def _norm(**kw):
    return NDVecNorm(in_keys=IN_KEYS, out_keys=OUT_KEYS, shapes=[3, 3], **kw)


def _raw(cfg, B, seed):
    obs = synthetic_obs(cfg, B, torch.Generator().manual_seed(seed))
    return {k: obs[k].to(G.dev()) for k in IN_KEYS}


# ---- 1. the kernels -----------------------------------------------------------------------------------------------------
def test_frozen_apply_equals_torch_call_bit_for_bit():
    """Same state -> torch's standardisation bit for bit; updating, `count` follows torch's bit for bit every step."""
    cfg = CONFIGS["rigid_insertion_multi_hepi_trpl_cfg"]
    dev_norm, torch_norm = _norm(), _norm()
    for step in range(6):
        raw = _raw(cfg, 64, 100 + step)
        td = dev_norm.apply_device(dict(raw))
        ref = torch_norm({k: v.view(v.shape[0], -1, 3) for k, v in raw.items()})
        for k in IN_KEYS:
            a, b = dev_norm._stats[k], torch_norm._stats[k]
            assert torch.equal(a["count"], b["count"]), f"step {step} {k}: count"
            assert G.rel(a["sum"], b["sum"]) <= 1e-6 and G.rel(a["ssq"], b["ssq"]) <= 1e-6
        for ok in OUT_KEYS:
            assert td[ok].shape == raw[IN_KEYS[OUT_KEYS.index(ok)]].shape
            assert G.rel(td[ok], ref[ok].reshape(td[ok].shape)) <= 1e-4
    # load the torch path's state into the device path: the same statistics give the same output, bit for bit
    dev_norm.load_state_dict(torch_norm.state_dict())
    dev_norm.freeze()
    torch_norm.freeze()
    raw = _raw(cfg, 64, 7)
    before = dev_norm.state_dict()
    got = dev_norm.apply_device(dict(raw))
    ref = torch_norm({k: v.view(v.shape[0], -1, 3) for k, v in raw.items()})
    for ok in OUT_KEYS:
        assert torch.equal(got[ok], ref[ok].reshape(got[ok].shape)), ok
    for k, v in dev_norm.state_dict().items():
        assert torch.equal(v, before[k]), f"frozen: {k} moved"


def _sizes():
    """(name, B, cfg) for M = 1, a ragged last slot and CTA, and every config's num_envs."""
    out = [("M=1", 1, None), ("ragged", 3, None)]
    out += [(n, CONFIGS[n].num_envs, CONFIGS[n]) for n in CONFIG_ORDER]
    return out


def _steps(B, cfg, n, seed):
    g = torch.Generator().manual_seed(seed)
    if cfg is None:  # M = 1: one position row, one velocity row; ragged: 3 x 601 and 3 x 7 rows
        F = (3, 3) if B == 1 else (3 * 601, 21)
        scale = torch.tensor([0.3, 2.0, 0.05])
        return [{k: (torch.randn(B, f // 3, 3, generator=g) * scale + 0.1).reshape(B, f).to(G.dev())
                 for k, f in zip(IN_KEYS, F)} for _ in range(n)]
    return [_raw(cfg, B, seed + i) for i in range(n)]


@pytest.mark.parametrize("name,B,cfg", _sizes(), ids=[s[0] for s in _sizes()])
def test_ten_steps_against_the_fp64_running_statistics(name, B, cfg):
    """Ten steps against tests/test_transforms.py's fp64 loop; outputs pre-filled with NaN.  The state stays within
    1e-6 (relative to its largest component) of torch `__call__`, and the standardised outputs within 1e-5 (relative to
    their largest magnitude) of the fp64 loop, or within 1.5x torch `__call__`'s own distance to it where that is
    larger.  The latter happens at M = 1: one row per step has variance 0, the std is clamped to sqrt(eps) = 0.01, and
    the fp32 state's rounding in `x - mean` is amplified a hundredfold, in torch's arithmetic as in the kernels'.
    Measured on one B200: state 3.1e-7 at worst (EMPN, 4096 x 97 rows); outputs 8.7e-7 at worst for M > 1 (ragged),
    1.6e-5 at M = 1, where torch `__call__` is off by 1.6e-5 as well."""
    decay, eps = 0.9999, 1e-4
    steps = _steps(B, cfg, 10, 900)
    dev_norm, torch_norm = _norm(decay=decay, eps=eps), _norm(decay=decay, eps=eps)
    ref = {k: _naive([s[k].view(B, -1, 3).cpu() for s in steps], decay, eps) for k in IN_KEYS}
    worst_state, worst_out, worst_torch = 0.0, 0.0, 0.0
    for i, raw in enumerate(steps):
        out = {ok: torch.full_like(raw[k], float("nan")) for k, ok in zip(IN_KEYS, OUT_KEYS)}
        dev_norm.apply_device(dict(raw), out=out)
        tout = torch_norm({k: v.view(B, -1, 3) for k, v in raw.items()})
        for k, ok in zip(IN_KEYS, OUT_KEYS):
            assert torch.isfinite(out[ok]).all(), f"step {i} {ok}: unwritten or non-finite entries"
            e_out = G.rel(out[ok], ref[k][i].reshape(B, -1))
            e_torch = G.rel(tout[ok], ref[k][i])
            a, b = dev_norm._stats[k], torch_norm._stats[k]
            assert torch.equal(a["count"], b["count"])
            e_state = max(G.rel(a["sum"], b["sum"]), G.rel(a["ssq"], b["ssq"]))
            worst_out, worst_state, worst_torch = max(worst_out, e_out), max(worst_state, e_state), max(worst_torch, e_torch)
            assert e_state <= 1e-6, f"step {i} {k}: state rel {e_state:.3e}"
            assert e_out <= max(1e-5, 1.5 * e_torch), f"step {i} {ok}: output rel {e_out:.3e} (torch {e_torch:.3e})"
    print(f"\n[obsnorm fp64] {name} B={B}: worst state rel {worst_state:.3e}, worst output rel {worst_out:.3e} "
          f"(torch __call__ {worst_torch:.3e})")


def test_results_do_not_change_with_an_sm_reservation():
    from geometry_rl_b200 import _lib as L
    cfg = CONFIGS["rigid_pushing_multi_empn_trpl_cfg"]
    steps = _steps(cfg.num_envs, cfg, 3, 50)
    res = []
    for reserve in (0, 4):
        L.reserve_sms(reserve)
        try:
            norm = _norm()
            outs = [norm.apply_device(dict(s)) for s in steps]
            res.append(([o[ok] for o in outs for ok in OUT_KEYS], norm.state_dict()))
        finally:
            L.reserve_sms(0)
    for a, b in zip(res[0][0], res[1][0]):
        assert torch.equal(a, b)
    for k in res[0][1]:
        assert torch.equal(res[0][1][k], res[1][1][k]), k


# ---- 2. the acting graph ------------------------------------------------------------------------------------------------
def _act_outs(td):
    return [td[k].clone() for k in ACT_KEYS + tuple(OUT_KEYS)]


def _without_norm_keys(td):
    return {k: v for k, v in td.items() if k not in OUT_KEYS}


def _states_equal(a, b):
    return a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)


@pytest.mark.parametrize("cfg_name", CONFIG_ORDER)
def test_graphed_equals_eager_for_every_config(cfg_name):
    from tests.test_gpu_act import SIZES, _agent, _obs_batches
    cfg, actor, _, _ = _agent(cfg_name)
    B, K = SIZES[cfg_name], 4
    obs = _obs_batches(cfg, B, K + 1, 300)
    norm = _norm()
    with torch.no_grad():
        actor.get_dist(norm.apply_device(dict(obs[0])))  # calibration + topology from a normalised first batch
    init = norm.state_dict()
    actor.set_act_state(1234, 0)
    eager = []
    for td in obs[1:]:
        td = norm.apply_device(dict(td))
        actor.act(td)
        eager.append(_act_outs(td))
    final = norm.state_dict()
    assert not _states_equal(final, init)

    norm.load_state_dict(init)
    actor.capture_act(obs[0], seed=1234, obs_norm=norm)
    assert _states_equal(norm.state_dict(), init), "capture moved the statistics"
    for i, (td, ref) in enumerate(zip(obs[1:], eager)):
        td = _without_norm_keys(td)
        actor.act_graphed(td)
        for name, got, exp in zip(ACT_KEYS + tuple(OUT_KEYS), _act_outs(td), ref):
            assert torch.equal(got, exp), f"step {i}: {name} graphed != eager"
    assert _states_equal(norm.state_dict(), final)
    assert actor.act_state() == (1234, K)

    # restored statistics: the replay reads them in place
    norm.load_state_dict(init)
    actor.set_act_state(1234, 0)
    td = actor.act_graphed(_without_norm_keys(obs[1]))
    for name, got, exp in zip(ACT_KEYS + tuple(OUT_KEYS), _act_outs(td), eager[0]):
        assert torch.equal(got, exp), f"after load_state_dict: {name}"

    # freezing after an updating capture: the graph would still update, so the replay refuses
    norm.freeze()
    with pytest.raises(RuntimeError, match="re-capture"):
        actor.act_graphed(_without_norm_keys(obs[1]))


def test_frozen_capture_never_moves_the_statistics():
    from tests.test_gpu_act import RIGID, SIZES, _agent, _obs_batches
    cfg, actor, _, _ = _agent(RIGID)
    obs = _obs_batches(cfg, SIZES[RIGID], 4, 500)
    norm = _norm()
    for td in obs:
        norm.apply_device(dict(td))
    with torch.no_grad():
        actor.get_dist(norm.apply_device(dict(obs[0])))
    norm.freeze()
    frozen = norm.state_dict()
    actor.capture_act(obs[0], seed=5, obs_norm=norm)
    for _ in range(2):
        for td in obs[1:]:
            got = actor.act_graphed(_without_norm_keys(td))
            ref = norm.apply_device(dict(td))
            for ok in OUT_KEYS:
                assert torch.equal(got[ok], ref[ok])
            assert _states_equal(norm.state_dict(), frozen)
    # restored statistics reach the frozen graph too
    other = _norm()
    other.apply_device(dict(obs[3]))
    norm.load_state_dict(other.state_dict())
    got = actor.act_graphed(_without_norm_keys(obs[1]))
    ref = norm.apply_device(dict(obs[1]))
    for ok in OUT_KEYS:
        assert torch.equal(got[ok], ref[ok])
    norm.frozen = False
    with pytest.raises(RuntimeError, match="re-capture"):
        actor.act_graphed(_without_norm_keys(obs[1]))


# ---- 3. two ranks, each holding half the environments -------------------------------------------------------------------
DP_CFG, DP_B, DP_K = "rigid_insertion_multi_hepi_trpl_cfg", 8, 3


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_obs():
    from tests.test_gpu_act import _obs_batches
    return _obs_batches(CONFIGS[DP_CFG], DP_B, DP_K + 1, 800)


def _dp_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from geometry_rl_b200.parallel import DataParallel
        from tests.test_gpu_act import _agent
        dev = torch.device("cuda", rank if torch.cuda.device_count() >= world else 0)
        torch.cuda.set_device(dev)
        _, actor, _, _ = _agent(DP_CFG)
        norm = _norm(dp=DataParallel())
        sl = slice(rank * DP_B // world, (rank + 1) * DP_B // world)
        obs = [{k: v[sl].to(dev) for k, v in td.items()} for td in _dp_obs()]
        with torch.no_grad():
            actor.get_dist(norm.apply_device(dict(obs[0])))
        init = norm.state_dict()
        actor.set_act_state(77, 0)
        eager, stats = [], []
        for td in obs[1:]:
            td = norm.apply_device(dict(td))
            actor.act(td)
            eager.append([t.cpu() for t in _act_outs(td)])
            stats.append({k: v.cpu() for k, v in norm.state_dict().items()})
        norm.load_state_dict(init)
        actor.capture_act(obs[0], seed=77, obs_norm=norm)
        graphed = []
        for td in obs[1:]:
            graphed.append([t.cpu() for t in _act_outs(actor.act_graphed(_without_norm_keys(td)))])
        final = {k: v.cpu() for k, v in norm.state_dict().items()}
        torch.cuda.synchronize()
        torch.save({"eager": eager, "graphed": graphed, "stats": stats, "final": final},
                   os.path.join(out_dir, f"rank{rank}.pt"))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_ranks_share_global_statistics(tmp_path):
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, str(tmp_path))) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    res = [torch.load(tmp_path / f"rank{r}.pt", weights_only=True) for r in range(world)]
    # the captured graph (split at the statistics all-reduce) equals the eager path on every rank
    for r in range(world):
        for i, (g, e) in enumerate(zip(res[r]["graphed"], res[r]["eager"])):
            for name, a, b in zip(ACT_KEYS + tuple(OUT_KEYS), g, e):
                assert torch.equal(a, b), f"rank {r} step {i}: {name} graphed != eager"
        assert _states_equal(res[r]["final"], res[r]["stats"][-1])
    # bit-identical statistics on both ranks, equal to one process over all environments within fp32 rounding
    single = _norm()
    obs = _dp_obs()
    single.apply_device(dict(obs[0]))
    for i, td in enumerate(obs[1:]):
        out = single.apply_device(dict(td))
        for k, v in single.state_dict().items():
            assert torch.equal(res[0]["stats"][i][k], res[1]["stats"][i][k]), f"step {i}: {k} differs between ranks"
            assert G.rel(res[0]["stats"][i][k], v) <= 1e-6, G.err_report(k, res[0]["stats"][i][k], v)
        for j, ok in enumerate(OUT_KEYS):
            got = torch.cat([res[r]["eager"][i][len(ACT_KEYS) + j] for r in range(world)], 0)
            assert G.rel(got, out[ok]) <= 1e-5, G.err_report(ok, got, out[ok])
