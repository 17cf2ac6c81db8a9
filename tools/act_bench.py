"""Time of one rollout-time policy call (the collector's `actor(td)` once per environment step) for each of the five
configs at that config's num_envs:

  eager_forward_ms   PolicyOperator.forward: body, torch head, torch.randn sampling, log_prob, diag_embed
  act_ms             PolicyOperator.act: body, then grl_gaussian_act + grl_act_advance, launched eagerly
  act_graphed_ms     PolicyOperator.act_graphed: observations copied into the static inputs, one CUDA-graph replay,
                     copies of the outputs
  kernel_us          grl_gaussian_act alone (torch.profiler device time per launch, a separate pass)

Each call time is the median over --regions regions of --calls calls, from CUDA events.  Observations are seeded
synthetic frames (geometry_rl_b200.synthetic), one batch of num_envs frames per config.  Prints one JSON object (card
name and power limit included) and writes it to --out.  Usage: python tools/act_bench.py --out profiles/r04_act.json"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:  # reporting only
        q = f"unavailable ({exc})"
    return q


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


def kernel_us(actor, td, calls):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            actor.act(dict(td))
        torch.cuda.synchronize()
    ev = [e for e in prof.key_averages() if "gaussian_act_kernel" in e.key]
    if not ev:
        raise RuntimeError("no gaussian_act_kernel launch in the profile")
    return sum(e.device_time_total for e in ev) / sum(e.count for e in ev)


def run_config(name, calls, regions, dev):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.synthetic import CONFIGS, synthetic_obs
    from geometry_rl_b200.tensors import to_device
    cfg = CONFIGS[name]
    B = cfg.num_envs
    actor, _, _, _, _ = learner.build_agent(cfg, dev, seed=0)
    td = to_device(synthetic_obs(cfg, B, torch.Generator().manual_seed(2024)), dev)
    with torch.no_grad():
        actor.get_dist(td)  # one-time calibration and the topology of this batch size
    res = {"num_envs": B, "k": cfg.total_action_dim}
    res["eager_forward_ms"] = timed(lambda: actor(dict(td)), calls, regions)
    actor.set_act_state(0, 0)
    res["act_ms"] = timed(lambda: actor.act(dict(td)), calls, regions)
    actor.capture_act(td, seed=0)
    res["act_graphed_ms"] = timed(lambda: actor.act_graphed(dict(td)), calls, regions)
    res["kernel_us"] = kernel_us(actor, td, calls)
    res["speedup_graphed_vs_eager"] = res["eager_forward_ms"] / res["act_graphed_ms"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50, help="calls per timed region")
    ap.add_argument("--regions", type=int, default=5, help="timed regions; the median is reported")
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16"])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("act_bench needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    from geometry_rl_b200 import ops
    from geometry_rl_b200.synthetic import CONFIG_ORDER
    ops.set_precision(args.precision)
    dev = torch.device("cuda:0")
    res = {"what": "one rollout-time policy call per environment step", "precision": args.precision, "card": card(),
           "calls": args.calls, "regions": args.regions, "configs": {}}
    for name in CONFIG_ORDER:
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
