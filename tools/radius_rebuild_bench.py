"""Step time of the rope policy update (rope_shaping_hepi_trpl_cfg, 16-bit fused path) with kNN and radius INTERNAL
edges, built once or rebuilt from the current positions on every step:

  knn_build_once            today's rope line (CUDA-graph replay)
  radius_build_once         radius graph of the first minibatch, kept (replay)
  radius_rebuild_graphed    radius graph refreshed in place inside the captured update (replay)
  radius_rebuild_eager      the same refresh mode, the update launched eagerly
  rebuild_only_graphed      the in-place refresh alone, captured and replayed

The edge kernels scale with the number of edges, so the mean INTERNAL degree is printed next to every time.  Prints one
JSON object (card name and power limit included) and writes it to --out.  Single process; data-parallel runs are not
covered here.  Usage: python tools/radius_rebuild_bench.py --out profiles/r03_radius_rebuild.json"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

NAME = "rope_shaping_hepi_trpl_cfg"


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:  # reporting only
        q = f"unavailable ({exc})"
    return q


def timed(fn, n, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def run_variant(internal, rebuild, graphed, B, steps, radius, max_nb, dev):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.synthetic import CONFIGS, synthetic_minibatch, synthetic_obs
    from geometry_rl_b200.tensors import to_device
    cfg = CONFIGS[NAME]
    actor, critic, _, loss_module, _ = learner.build_agent(cfg, dev, seed=0)
    hd = actor.get_submodule("0").module.hyper_data
    if internal == "radius":
        hd.internal_edges, hd.radius, hd.max_num_neighbors = "radius", radius, max_nb
    hd.rebuild_every_call = rebuild
    gen = torch.Generator().manual_seed(4321)
    mbs = []
    for s in range(4):  # the rope moves between minibatches
        obs = synthetic_obs(cfg, B, gen, env_ids=(torch.arange(B) + s) % cfg.num_envs)
        if not mbs:
            actor.get_dist(to_device(obs, dev))  # one-time calibration
        with torch.no_grad():
            d_ = actor.get_dist(to_device(obs, dev))
            v = critic.module(*[obs[k].to(dev) for k in critic.in_keys])
        mbs.append(to_device(synthetic_minibatch(obs, d_.mean, d_.var_diag, v, gen), dev))
    lrn = learner.Learner(cfg, actor, critic, loss_module)
    it = [0]

    if graphed:
        lrn.capture(mbs[0])

        def step():
            it[0] += 1
            return lrn.update_graphed(mbs[it[0] % len(mbs)])
    else:
        def step():
            it[0] += 1
            return lrn.update(mbs[it[0] % len(mbs)])

    ms = timed(step, steps)
    es = hd.example_data.edge_sets[("links", "internal", "links")]
    n_links = hd.example_data.nodes_per_graph["links"] * B
    out = {"ms_per_step": ms, "samples_per_s": B / (ms * 1e-3),
           "mean_internal_degree": int(es.rowptr_dst[-1]) / n_links,
           "internal_edge_capacity": es.n_edges if not es.exact else None}
    if graphed and rebuild:
        pol = [mbs[1][k] for k in actor.in_keys]
        hd.build_data(*pol, train=True)
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            hd.build_data(*pol, train=True)
        torch.cuda.current_stream().wait_stream(s)
        with torch.cuda.graph(g):
            hd.build_data(*pol, train=True)
        out["rebuild_only_graphed_ms"] = timed(g.replay, steps)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--minibatch", type=int, default=2048)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--radius", type=float, default=0.025)
    ap.add_argument("--max-num-neighbors", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("radius_rebuild_bench needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    from geometry_rl_b200 import ops
    ops.set_precision("bf16")
    dev = torch.device("cuda:0")
    res = {"workload": f"{NAME}@{args.minibatch}", "precision": "bf16 (fused edge path)", "card": card(),
           "radius": args.radius, "max_num_neighbors": args.max_num_neighbors, "knn_k": 3, "steps": args.steps}
    variants = {"knn_build_once": ("knn", False, True), "radius_build_once": ("radius", False, True),
                "radius_rebuild_graphed": ("radius", True, True), "radius_rebuild_eager": ("radius", True, False)}
    for key, (internal, rebuild, graphed) in variants.items():
        res[key] = run_variant(internal, rebuild, graphed, args.minibatch, args.steps, args.radius,
                               args.max_num_neighbors, dev)
        print(key, json.dumps(res[key]), flush=True)
    res["rebuild_only_graphed_ms"] = res["radius_rebuild_graphed"].pop("rebuild_only_graphed_ms")
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
