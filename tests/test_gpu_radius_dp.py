"""GPU: data-parallel update step with the radius topology refreshed in place on every call (16-bit fused path) ==
the single-process step on the whole minibatch.  Two ranks (gloo rendezvous, as in test_gpu_dp.py) each rebuild the
radius graph of their half of the minibatch; losses and all-reduced gradients within the 16-bit bound (1e-2)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
CFG = "rope_shaping_hepi_trpl_cfg"
B = 8
KEYS = ("loss_objective", "loss_trust_region", "loss_entropy", "loss_critic", "ESS", "kl", "constraint", "mean_constraint",
        "mean_constraint_max", "cov_constraint", "cov_constraint_max", "entropy", "entropy_diff")


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _setup(dev):
    from geometry_rl_b200 import learner, ops
    from geometry_rl_b200.tensors import to_device
    from geometry_rl_b200.synthetic import CONFIGS, synthetic_minibatch, synthetic_obs
    ops.set_precision("bf16")
    cfg = CONFIGS[CFG]
    actor, critic, _, loss_module, _ = learner.build_agent(cfg, dev, seed=0)
    hd = actor.get_submodule("0").module.hyper_data
    hd.internal_edges, hd.radius, hd.max_num_neighbors = "radius", 0.025, 8
    hd.rebuild_every_call = True
    assert hd.refresh_in_place()
    gen = torch.Generator().manual_seed(78)
    obs = synthetic_obs(cfg, B, gen, env_ids=torch.arange(B) * (cfg.num_envs // B))
    with torch.no_grad():  # calibration on the FULL batch in every process -> identical replicas
        d = actor.get_dist(to_device(obs, dev))
        v = critic.module(*[obs[k].to(dev) for k in critic.in_keys])
    mb = synthetic_minibatch(obs, d.mean, d.var_diag, v, gen)
    return cfg, actor, critic, loss_module, mb


def _grads(actor, critic):
    return [p.grad.detach().cpu().clone() if p.grad is not None else None
            for p in list(actor.parameters()) + list(critic.parameters())]


def _worker(rank, world, port, out_path):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from geometry_rl_b200 import learner
        from geometry_rl_b200.parallel import DataParallel
        from geometry_rl_b200.tensors import to_device
        dev = torch.device("cuda", rank if torch.cuda.device_count() >= world else 0)
        torch.cuda.set_device(dev)
        cfg, actor, critic, loss_module, mb = _setup(dev)
        dp = DataParallel()
        lrn = learner.Learner(cfg, actor, critic, loss_module, dp=dp)
        sl = slice(rank * B // world, (rank + 1) * B // world)
        shard = {k: (v[sl] if torch.is_tensor(v) else v) for k, v in mb.items()}
        out = lrn.compute_losses(to_device(shard, dev))
        out["actor_loss"].backward()
        out["loss_critic"].backward()
        dp.allreduce_grads(list(actor.parameters()) + list(critic.parameters()))
        logged = dp.global_losses(out)
        torch.cuda.synchronize()
        if rank == 0:
            torch.save({"losses": {k: logged[k].detach().cpu() for k in KEYS}, "grads": _grads(actor, critic)}, out_path)
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_rank_step_with_radius_rebuild_equals_single_process(tmp_path):
    from geometry_rl_b200 import learner, ops
    from geometry_rl_b200.tensors import to_device
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    out_path = str(tmp_path / "rank0.pt")
    procs = [ctx.Process(target=_worker, args=(r, world, port, out_path)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    res = torch.load(out_path, weights_only=True)
    try:
        dev = torch.device("cuda:0")
        cfg, actor, critic, loss_module, mb = _setup(dev)
        lrn = learner.Learner(cfg, actor, critic, loss_module)
        out = lrn.compute_losses(to_device(mb, dev))
        out["actor_loss"].backward()
        out["loss_critic"].backward()
        bad = []
        for k in KEYS:
            a, b = float(res["losses"][k]), float(out[k])
            tol = 1e-2 if k == "loss_objective" else 1e-2 * abs(b) + 1e-5
            if not abs(a - b) <= tol:
                bad.append(f"{k}: dp {a} vs single {b}")
        for i, (g_dp, g1) in enumerate(zip(res["grads"], _grads(actor, critic))):
            if g1 is None or float(g1.abs().max()) == 0.0:
                continue
            err = float((g_dp - g1).abs().max()) / float(g1.abs().max())
            if not err <= 1e-2:
                bad.append(f"grad[{i}] rel err {err:.2e}")
        assert not bad, "\n".join(bad)
    finally:
        ops.set_precision("fp32")
