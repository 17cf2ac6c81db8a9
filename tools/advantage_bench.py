"""Time and peak memory of the advantage phase (`adv_module(data)`, once per rollout) for each of the five configs at that
config's num_envs x rollout_len:

  forward_ms           GAE.forward: the torch formulation of the critic's per-token half ([tokens, 64] activations)
  advantage_ms         GAE.advantage: the per-token half on grl_critic_inner_stats / _fwd with per-time-step statistics
  advantage_graphed_ms GAE.advantage_graphed: inputs copied into the static [B_env, T+1, F] buffers, one replay, copies
  kernels_ms           the grouped grl_critic_inner_stats + _fwd alone on the phase's [B_env (T+1), N, F] tokens

Each time is the median over --regions regions of --calls calls, from CUDA events, after warm-up.  `*_peak_bytes` is
torch.cuda.max_memory_allocated over that mode's calls and `*_extra_bytes` the same less what was allocated before them
(the rollout, the model and, for the graphed mode, the graph's static buffers).  Inputs are seeded synthetic rollouts
(geometry_rl_b200.synthetic).  Prints one JSON object (card name, power limit and max SM clock included) and writes it
to --out.  Usage: python tools/advantage_bench.py --out profiles/r06_advantage.json"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.act_bench import card  # noqa: E402


def timed(fn, calls, regions, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = []
    for _ in range(regions):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(calls):
            fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b) / calls)
    peak = torch.cuda.max_memory_allocated()
    return statistics.median(out), peak, peak - base


def rollout_td(cfg, keys, dev):
    from geometry_rl_b200.synthetic import synthetic_rollout
    roll = synthetic_rollout(cfg, torch.Generator().manual_seed(2024))
    td = {k: roll[k][:, :-1].to(dev) for k in keys}
    td["next"] = {k: roll[k][:, 1:].to(dev) for k in keys}
    td["next"].update({"reward": roll["reward"].unsqueeze(-1).to(dev), "done": roll["done"].unsqueeze(-1).to(dev),
                       "terminated": roll["terminated"].unsqueeze(-1).to(dev)})
    return td


def fresh(td):
    out = {k: v for k, v in td.items() if k != "next"}
    out["next"] = dict(td["next"])
    return out


def tokens(critic, td):
    """The [B_env (T+1), N, F] token tensor of the phase, time-major, as DeepSets.one_step builds it."""
    vf = critic.module._network1
    obs = [torch.cat([td[k], td["next"][k][:, -1:]], dim=1) for k in critic.in_keys]
    B, T1, _ = obs[0].shape
    flat = [a.transpose(0, 1).reshape(T1 * B, a.shape[-1]) for a in obs]
    with torch.no_grad():
        data, iv = vf.hyper_data.build_data(*flat, train=True)
        x = torch.cat([iv[t].reshape(T1 * B, -1, iv[t].shape[-1]) for t in data.node_types], dim=1).contiguous()
    return x, T1


def run_config(name, calls, regions, dev):
    from geometry_rl_b200 import learner, ops
    from geometry_rl_b200.synthetic import CONFIGS
    cfg = CONFIGS[name]
    _, critic, _, _, adv = learner.build_agent(cfg, dev, seed=0)
    td = rollout_td(cfg, critic.in_keys, dev)
    res = {"num_envs": cfg.num_envs, "rollout_len": cfg.rollout_len, "graphs": cfg.num_envs * (cfg.rollout_len + 1)}
    for mode, fn in (("forward", lambda: adv(fresh(td))), ("advantage", lambda: adv.advantage(fresh(td)))):
        res[f"{mode}_ms"], res[f"{mode}_peak_bytes"], res[f"{mode}_extra_bytes"] = timed(fn, calls, regions)
    a, b = adv(fresh(td)), adv.advantage(fresh(td))
    res["max_rel_diff_advantage_vs_forward"] = float((a["advantage"] - b["advantage"]).abs().max()
                                                     / a["advantage"].abs().max())
    adv.capture(td)
    res["advantage_graphed_ms"], res["advantage_graphed_peak_bytes"], res["advantage_graphed_extra_bytes"] = timed(
        lambda: adv.advantage_graphed(fresh(td)), calls, regions)
    x, T1 = tokens(critic, td)
    inner = critic.module._network1.gnn.mlp_inner
    norm = inner.norms[0]
    res["tokens_per_graph"], res["features"] = x.shape[1], x.shape[2]
    with torch.no_grad():
        res["kernels_ms"], _, _ = timed(lambda: ops.critic_inner(x, inner.lins[0].weight, inner.lins[0].bias, norm.weight,
                                                                 norm.bias, norm.eps, groups=T1), calls, regions)
    res["speedup_advantage_vs_forward"] = res["forward_ms"] / res["advantage_ms"]
    res["speedup_graphed_vs_forward"] = res["forward_ms"] / res["advantage_graphed_ms"]
    del adv, critic, td, x
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5, help="calls per timed region")
    ap.add_argument("--regions", type=int, default=3, help="timed regions; the median is reported")
    ap.add_argument("--config", action="append", default=None, help="config name (repeatable; default: all five)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("advantage_bench needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    from geometry_rl_b200.synthetic import CONFIG_ORDER
    dev = torch.device("cuda:0")
    res = {"what": "advantage phase, one call per rollout, each config at num_envs x rollout_len", "card": card(),
           "calls": args.calls, "regions": args.regions, "configs": {}}
    for name in args.config or CONFIG_ORDER:
        res["configs"][name] = run_config(name, args.calls, args.regions, dev)
        print(name, json.dumps(res["configs"][name]), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
