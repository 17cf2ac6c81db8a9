"""Step time of the policy update with kNN INTERNAL edges (k = 3) built once or rebuilt from the current positions on
every step, for rope (rope_shaping_hepi_trpl_cfg) and rigid insertion (rigid_insertion_multi_hepi_trpl_cfg):

  knn_build_once         the reference's build-once rule (16-bit fused path, CUDA-graph replay)
  knn_rebuild_graphed    kNN set rebuilt in place inside the captured update (knn_in_place; 16-bit, replay)
  knn_rebuild_eager      today's eager exact-size rebuild (rebuild_every_call without knn_in_place; 16-bit, `update`)
  rebuild_only_graphed   the in-place refresh alone (build_data of the policy graph), captured and replayed
  knn_rebuild_graphed_fp32  rope only: the in-place rebuild on the strict fp32 path (exact-size set, replay)

and for the EMPN policy (rigid_pushing_multi_empn_trpl_cfg), whose in-place rebuild also merges the homogeneous view and
the last layer's sub set on the device (GraphBatch.refresh_homogeneous), the first four.

Prints one JSON object (card name and power limit included) and writes it to --out.  Single process; data-parallel runs
are not covered here.  Usage: python tools/knn_rebuild_bench.py --out profiles/r04_knn_rebuild.json"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.radius_rebuild_bench import card, timed  # noqa: E402

WORKLOADS = {"rope_shaping_hepi_trpl_cfg": 2048, "rigid_insertion_multi_hepi_trpl_cfg": 8192,
             "rigid_pushing_multi_empn_trpl_cfg": 4096}


def run_variant(name, B, steps, rebuild, in_place, graphed, precision, dev):
    from geometry_rl_b200 import learner, ops
    from geometry_rl_b200.synthetic import CONFIGS, synthetic_minibatch, synthetic_obs
    from geometry_rl_b200.tensors import to_device
    ops.set_precision(precision)
    cfg = CONFIGS[name]
    actor, critic, _, loss_module, _ = learner.build_agent(cfg, dev, seed=0)
    hd = actor.get_submodule("0").module.hyper_data
    hd.rebuild_every_call, hd.knn_in_place = rebuild, in_place
    assert hd.refresh_in_place() == (rebuild and in_place)
    gen = torch.Generator().manual_seed(4321)
    mbs = []
    for s in range(4):  # the positions move between minibatches
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
    out = {"ms_per_step": ms, "samples_per_s": B / (ms * 1e-3)}
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
    ops.set_precision("fp32")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rope-minibatch", type=int, default=WORKLOADS["rope_shaping_hepi_trpl_cfg"])
    ap.add_argument("--rigid-minibatch", type=int, default=WORKLOADS["rigid_insertion_multi_hepi_trpl_cfg"])
    ap.add_argument("--empn-minibatch", type=int, default=WORKLOADS["rigid_pushing_multi_empn_trpl_cfg"])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("knn_rebuild_bench needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda:0")
    res = {"card": card(), "knn_k": 3, "steps": args.steps, "precision": "bf16 (fused edge path) unless noted"}
    variants = {"knn_build_once": (False, False, True, "bf16"), "knn_rebuild_graphed": (True, True, True, "bf16"),
                "knn_rebuild_eager": (True, False, False, "bf16")}
    for name, B in (("rope_shaping_hepi_trpl_cfg", args.rope_minibatch),
                    ("rigid_insertion_multi_hepi_trpl_cfg", args.rigid_minibatch),
                    ("rigid_pushing_multi_empn_trpl_cfg", args.empn_minibatch)):
        cur = res[f"{name}@{B}"] = {}
        todo = dict(variants)
        if name.startswith("rope"):
            todo["knn_rebuild_graphed_fp32"] = (True, True, True, "fp32")
        for key, (rebuild, in_place, graphed, precision) in todo.items():
            cur[key] = run_variant(name, B, args.steps, rebuild, in_place, graphed, precision, dev)
            print(name, key, json.dumps(cur[key]), flush=True)
        cur["rebuild_only_graphed_ms"] = cur["knn_rebuild_graphed"].pop("rebuild_only_graphed_ms")
        if "knn_rebuild_graphed_fp32" in cur:
            cur["rebuild_only_graphed_fp32_ms"] = cur["knn_rebuild_graphed_fp32"].pop("rebuild_only_graphed_ms")
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
