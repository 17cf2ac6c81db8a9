"""Time of one collection step's observation normalisation plus acting for each of the five configs at that config's
num_envs (one acting call per environment step):

  torch_call_act_graphed_ms  NDVecNorm.__call__ (the torch restatement, on the [B, n, 3] views) writing the norm_* keys,
                             then PolicyOperator.act_graphed captured without a normaliser (it copies the norm_* keys in)
  act_graphed_obs_norm_ms    act_graphed captured with obs_norm: the raw groups are copied in and one replay runs the
                             statistics update, the standardisation and the policy
  apply_device_ms            NDVecNorm.apply_device alone (the four grl_vecnorm launches, eager)
  kernels_us                 the grl_vecnorm kernels alone from torch.profiler (device time per call, summed per kernel name,
                             over --profile-calls eager apply_device calls, in a separate profiled pass)

Each time is the median over --regions regions of --calls calls, from CUDA events, after warm-up; the statistics keep
updating during the timed calls (decay 0.9999, as configured).  Inputs are seeded synthetic observations
(geometry_rl_b200.synthetic).  Prints one JSON object (card name, power limit and max SM clock included) and writes it to
--out.  Usage: python tools/obs_norm_bench.py --out profiles/r07_obs_norm.json"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.act_bench import card  # noqa: E402
from tools.advantage_bench import timed  # noqa: E402

IN_KEYS = ["position_vectors", "velocity_vectors"]
OUT_KEYS = ["norm_position_vectors", "norm_velocity_vectors"]


def make_norm():
    from geometry_rl_b200.torchrl.envs import NDVecNorm
    return NDVecNorm(in_keys=IN_KEYS, out_keys=OUT_KEYS, shapes=[3, 3], decay=0.9999, eps=1e-4)


def torch_norm_step(norm, td):
    """The eager collector step: __call__ on the reshaped views, the norm_* keys handed on in the env's flat layout."""
    views = {k: td[k].view(td[k].shape[0], -1, 3) for k in IN_KEYS}
    norm(views)
    for ok in OUT_KEYS:
        td[ok] = views[ok].reshape(td[ok].shape)
    return td


def kernel_times(fn, calls):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if "vecnorm" in e.key:
            t = getattr(e, "self_device_time_total", None)
            if t is None:
                t = e.self_cuda_time_total
            out[e.key] = t / calls
    return out


def run_config(name, calls, regions, profile_calls, dev):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.synthetic import CONFIGS, synthetic_obs
    from geometry_rl_b200.tensors import to_device
    cfg = CONFIGS[name]
    B = cfg.num_envs
    actor, _, _, _, _ = learner.build_agent(cfg, dev, seed=0)
    env_ids = torch.arange(B)
    obs = to_device(synthetic_obs(cfg, B, torch.Generator().manual_seed(2024), env_ids=env_ids), dev)
    res = {"num_envs": B, "rows": {k: B * obs[k].shape[1] // 3 for k in IN_KEYS}}
    norm = make_norm()
    with torch.no_grad():
        actor.get_dist(norm.apply_device(dict(obs)))  # calibration + topology
    start = norm.state_dict()

    actor.capture_act(obs, seed=1)
    torch_norm = make_norm()
    torch_norm.load_state_dict(start)
    res["torch_call_act_graphed_ms"], _, _ = timed(lambda: actor.act_graphed(torch_norm_step(torch_norm, dict(obs))),
                                                   calls, regions)
    res["apply_device_ms"], _, _ = timed(lambda: norm.apply_device(dict(obs)), calls, regions)
    norm.load_state_dict(start)
    actor.capture_act(obs, seed=1, obs_norm=norm)
    raw = {k: v for k, v in obs.items() if k not in OUT_KEYS}
    res["act_graphed_obs_norm_ms"], _, _ = timed(lambda: actor.act_graphed(dict(raw)), calls, regions)
    res["speedup"] = res["torch_call_act_graphed_ms"] / res["act_graphed_obs_norm_ms"]
    res["kernels_us"] = kernel_times(lambda: norm.apply_device(dict(obs)), profile_calls)
    res["kernels_total_us"] = sum(res["kernels_us"].values())
    del actor, norm, torch_norm, obs, raw
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20, help="calls per timed region")
    ap.add_argument("--regions", type=int, default=5, help="timed regions; the median is reported")
    ap.add_argument("--profile-calls", type=int, default=50)
    ap.add_argument("--config", action="append", default=None, help="config name (repeatable; default: all five)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("obs_norm_bench needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    from geometry_rl_b200.synthetic import CONFIG_ORDER
    dev = torch.device("cuda:0")
    res = {"what": "observation normalisation + acting, one collection step, each config at num_envs", "card": card(),
           "calls": args.calls, "regions": args.regions, "configs": {}}
    for name in args.config or CONFIG_ORDER:
        res["configs"][name] = run_config(name, args.calls, args.regions, args.profile_calls, dev)
        print(name, json.dumps(res["configs"][name]), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
