"""Cost of TRPL entropy control in the update step, per config (HEPi rigid insertion at minibatch 8192 and HEPi rope at
its benchmark minibatch by default, 16-bit path as bench.py runs it):

  off_graphed_ms        entropy control off, Learner.capture + update_graphed (the default path)
  on_graphed_ms         entropy control on (linear schedule, inequality, after the trust-region projection), fused loss,
                        captured: the bound and the entropy projection run on the device inside the replay
  on_eager_unfused_ms   entropy control on, eager update with TRPLLoss.fused = False (the torch formulation)
  kernel_*_us           the kernels alone on the minibatch's [B, k] (CUDA events over --kernel-calls launches):
                        grl_trpl_entropy_bound (stage 0), grl_trpl_fwd / _bwd without and with entropy control

Step times are the median over --regions regions of --steps updates, from CUDA events, after warm-up, inputs resident
in HBM and rotated over two minibatches.  Prints one JSON object (card name, power limit and max SM clock included) and
writes it to --out.  Usage: python tools/entropy_control_bench.py --out profiles/r08_entropy_control.json"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.act_bench import card  # noqa: E402

CONFIGS = {"rigid_insertion_multi_hepi_trpl_cfg": 8192, "rope_shaping_hepi_trpl_cfg": 1024}
ENTROPY = dict(entropy_schedule="linear", target_entropy=-1.0, total_train_steps=1000)


def timed(fn, calls, regions, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(regions):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(calls):
            fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b) / calls)
    return statistics.median(out)


def batches(cfg, B, dev):
    from geometry_rl_b200.synthetic import synthetic_minibatch, synthetic_obs
    from geometry_rl_b200.tensors import to_device
    gen = torch.Generator().manual_seed(1234)
    out = []
    for _ in range(2):
        obs = synthetic_obs(cfg, B, gen, env_ids=torch.arange(B) * max(1, cfg.num_envs // B) % cfg.num_envs)
        k = cfg.total_action_dim  # bench.py's nominal old policy: the initial Gaussian head (mean 0, variance 1)
        out.append(to_device(synthetic_minibatch(obs, torch.zeros(B, k), torch.ones(B, k), torch.zeros(B, 1), gen), dev))
    return out


def step_ms(name, B, dev, steps, regions, entropy, graphed, fused=True):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.synthetic import CONFIGS as ALL
    cfg = ALL[name]
    actor, critic, _, loss_module, _ = learner.build_agent(cfg, dev, seed=0, projection_kwargs=ENTROPY if entropy else None)
    loss_module.fused = fused
    lrn = learner.Learner(cfg, actor, critic, loss_module)
    mbs = batches(cfg, B, dev)
    lrn.calibrate(mbs[0])
    i = [0]
    if graphed:
        lrn.capture(mbs[0], warmup=3)

        def fn():
            lrn.update_graphed(mbs[i[0] % 2])
            i[0] += 1
    else:
        def fn():
            lrn.update(mbs[i[0] % 2])
            i[0] += 1
    ms = timed(fn, steps, regions)
    del lrn, actor, critic, loss_module, mbs
    torch.cuda.empty_cache()
    return ms


def kernel_us(B, k, dev, calls, regions):
    """grl_trpl_entropy_bound and grl_trpl_fwd / _bwd (KL) on one [B, k] minibatch, without and with entropy control."""
    from geometry_rl_b200 import _lib as L, ops
    g = torch.Generator().manual_seed(3)
    q_mean = (torch.randn(B, k, generator=g) * 0.3).to(dev)
    q_v = ((0.5 + torch.rand(B, k, generator=g)) ** 2).to(dev)
    mean = q_mean + (torch.randn(B, k, generator=g) * 0.3).to(dev)
    v = q_v * torch.exp(torch.randn(B, k, generator=g) * 0.2).to(dev)
    pm, pv, gm, gv = (torch.empty(B, k, device=dev) for _ in range(4))
    g_pm, g_pv = (torch.randn(B, k, generator=g).to(dev) for _ in range(2))
    eta = torch.empty(B, 2, dtype=torch.float64, device=dev)
    alpha = torch.empty(B, dtype=torch.float64, device=dev)
    ent = ops.EntropyControl(torch.zeros(4, dtype=torch.float64, device=dev), torch.zeros((), dtype=torch.int64, device=dev),
                             "linear", 1000, -1.0, 0.5, False, False)
    # linear schedule at step 0: the bound is the mean old entropy, so part of the minibatch is projected
    res = {"kernel_entropy_bound_us": 1e3 * timed(lambda: ops.entropy_bound(ent, q_v), calls, regions)}
    for tag, mode in (("off", 0), ("on", L.ENTROPY_MODE["ineq"])):
        d = L.GrlProjDesc(batch=B, k=k, proj_type=0, eps_mean=0.05, eps_cov=0.0025, mean=L.ptr(mean), v=L.ptr(v),
                          old_mean=L.ptr(q_mean), old_v=L.ptr(q_v), proj_mean=L.ptr(pm), proj_v=L.ptr(pv), eta=L.ptr(eta),
                          grad_proj_mean=L.ptr(g_pm), grad_proj_v=L.ptr(g_pv), grad_mean=L.ptr(gm), grad_v=L.ptr(gv),
                          entropy_mode=mode, entropy_beta=L.ptr(ent.state[2:3]) if mode else None,
                          entropy_alpha=L.ptr(alpha) if mode else None)
        res[f"kernel_trpl_fwd_{tag}_us"] = 1e3 * timed(lambda: L.call("grl_trpl_fwd", C.byref(d)), calls, regions)
        res[f"kernel_trpl_bwd_{tag}_us"] = 1e3 * timed(lambda: L.call("grl_trpl_bwd", C.byref(d)), calls, regions)
    res["entropy_active_fraction"] = float((alpha > 1.0).double().mean())
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="updates per timed region")
    ap.add_argument("--regions", type=int, default=3, help="timed regions; the median is reported")
    ap.add_argument("--kernel-calls", type=int, default=200)
    ap.add_argument("--config", action="append", default=None, help="config name (repeatable; default: two configs)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("entropy_control_bench needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    from geometry_rl_b200 import ops
    from geometry_rl_b200.synthetic import CONFIGS as ALL
    ops.set_precision("bf16")
    dev = torch.device("cuda:0")
    res = {"what": "update step with TRPL entropy control (linear schedule, inequality, after the projection), 16-bit "
                   "path, one GPU", "card": card(), "steps": args.steps, "regions": args.regions, "configs": {}}
    for name in args.config or list(CONFIGS):
        B = CONFIGS.get(name, 1024)
        r = {"minibatch": B, "action_dim": ALL[name].total_action_dim}
        r["off_graphed_ms"] = step_ms(name, B, dev, args.steps, args.regions, False, True)
        r["on_graphed_ms"] = step_ms(name, B, dev, args.steps, args.regions, True, True)
        r["on_eager_unfused_ms"] = step_ms(name, B, dev, args.steps, args.regions, True, False, fused=False)
        r.update(kernel_us(B, ALL[name].total_action_dim, dev, args.kernel_calls, args.regions))
        res["configs"][name] = r
        print(name, json.dumps(r), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
