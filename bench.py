#!/usr/bin/env python
"""bench.py — policy-update throughput of the B200-native GeometryRL hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--dump-outputs DIR]

A "step" is one minibatch iteration of examples/torchrl/train.py:259-316 on synthetic rollout frames of the
config's graph shape: policy forward (graph features -> EMPN/HEPi/transformer -> Gaussian head), TRPL
projection, TRPLLoss, DeepSets critic forward, both backward passes, (DP: one NCCL gradient all-reduce),
optional grad-norm clip, two Adam steps.  Prints ONE JSON line (see the task contract): `value` = samples/s
with minibatches resident in HBM (default workload: the HEPi headline config, BASELINE.md section 4), `e2e` = the same
step fed from pinned HOST memory with a loss read back, `roofline` = the dominant kernel's algorithmic bytes (SURVEY
8(d) accounting) / CUDA-event duration against MEASURED_PEAKS.json, `cpu_baseline` = the CPU oracle port of the same
step on this box's host cores (bounded sample), `configs` = the other message-passing workloads, device-timed.

The minibatches are drawn from fixed seeds on the host without running the model (`nominal_policy_output`), so every
build of the project times and computes on the same inputs.  The starting parameters are seeded too, then calibrated
by the policy's first training-mode forward, which runs the kernels under test (the reference's conv.py:104-105 rule).

`--dump-outputs DIR` writes, as .npy files, the parameters the timed path started from right after that calibration
(`init.<actor|critic>.<parameter>.npy`) and what its last timed step produced: the losses and metrics it returns
(`out.<name>.npy`), the gradients it applied (`grad.<actor|critic>.<parameter>.npy`) and the parameters it left
(`param.<actor|critic>.<parameter>.npy`).  Two builds run with the same arguments can be compared file by file; equal
`init.*` files confirm that they started from the same state.

`--impl reference` times that CPU port alone (the reference itself is pure Python on top of torchrl / PyG /
ITPAL wheels that are not installable offline, so it cannot run unmodified here; see DESIGN.md)."""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# BASELINE.json's metric is "HEPi fwd+bwd+TRPL update samples/sec" and BASELINE.md section 4 names config 1
# (rigid_insertion_multi_hepi_trpl_cfg) as the headline; the other message-passing configs are reported in the same
# JSON line under "configs".
DEFAULT_CONFIG = "rigid_insertion_multi_hepi_trpl_cfg"
# Samples per GPU per step.  The config's own mini_batch_size (1000, configs/rigid_insertion_multi_hepi_trpl_cfg.yaml:138)
# is launch/latency-bound on a B200 (2.3 ms per step, every kernel a fraction of a wave); the headline fills the machine with
# 8192 graphs per step (8 of the reference's minibatches: its 1000 x 100 rollout holds 12 such steps per epoch) and the
# config's own size is reported next to it (configs["...@1000"]).
DEFAULT_MINIBATCH = {"rigid_insertion_multi_hepi_trpl_cfg": 8192, "rigid_pushing_multi_empn_trpl_cfg": 4096,
                     "cloth_hanging_multi_hepi_trpl_cfg": 8192, "rope_shaping_hepi_trpl_cfg": 2048}
# workloads reported under "configs" next to the headline: (config, samples per GPU per step)
SIDE_WORKLOADS = [("rigid_insertion_multi_hepi_trpl_cfg", 1000), ("rigid_pushing_multi_empn_trpl_cfg", 4096),
                  ("cloth_hanging_multi_hepi_trpl_cfg", 8192), ("rope_shaping_hepi_trpl_cfg", 2048),
                  ("rigid_insertion_two_agents_multi_transformer_trpl_cfg", 1000)]
METRIC = "fwd+bwd+TRPL update samples/sec (policy fwd+bwd, TRPL projection, losses, critic, Adam)"  # BASELINE.json metric
N_ROTATE = 8  # distinct minibatches cycled through the timed region
_emit = print


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps per region")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=DEFAULT_CONFIG)
    ap.add_argument("--minibatch", type=int, default=0, help="samples per GPU per step (default: DEFAULT_MINIBATCH, else the config's)")
    ap.add_argument("--no-side-workloads", action="store_true", help="skip the other configs reported under \"configs\"")
    ap.add_argument("--repeats", type=int, default=1, help="timed regions of --steps steps each; the median region is reported")
    ap.add_argument("--cpu-sample", type=int, default=256, help="samples per CPU-baseline step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-dp-graph", action="store_true", help="N > 1: launch the step eagerly instead of replaying it "
                    "(NCCL all-reduces included) from a CUDA graph")
    ap.add_argument("--dp-graph", action="store_true", help=argparse.SUPPRESS)  # now the default
    ap.add_argument("--no-dp-overlap", action="store_true", help="N > 1: keep the critic branch on the actor's stream "
                    "(default: second stream with its own NCCL communicator)")
    ap.add_argument("--single-precision", action="store_true", help="skip the second (other precision) measurement")
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16"],
                    help="nn.Linear contractions of the message-passing kernels: fp32 FFMA (parity 1e-5) or bf16 tcgen05 "
                         "tensor cores (parity 1e-2)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of the headline workload to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.repeats < 1 or args.warmup < 0:
        ap.error("--steps and --repeats must be at least 1, --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons of EVERY GPU of the job, sampled every 50 ms while the timed region runs (rank 0
    samples for all local ranks: under data parallelism the step time is the slowest rank's, so one power-capped GPU
    explains a scaling loss that rank 0's own clocks would hide)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, indices):
        self.indices = [int(i) for i in (indices if isinstance(indices, (list, tuple, range)) else [indices])]
        self.proc, self.lines = None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", ",".join(str(i) for i in self.indices), "-lms", "50"],
                                         stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        per_gpu, mx, reasons = {}, None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                per_gpu.setdefault(int(f[0]), []).append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        med = {g: sorted(v)[len(v) // 2] for g, v in per_gpu.items() if v}
        out = {"sm_mhz": min(med.values()) if med else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
               "samples": sum(len(v) for v in per_gpu.values())}
        if len(med) > 1:
            out["sm_mhz_per_gpu"] = [med[g] for g in sorted(med)]  # median under load, one entry per GPU of the job
        return out


def measured_traffic(kernel, workload, minibatch):
    """DRAM bytes per launch of `kernel` (dram__bytes_read.sum + dram__bytes_write.sum) from the committed
    `ncu --set full` capture of this same workload (profiles/r02_traffic.json, written by profiles/summarise.py
    traffic); None when no capture matches the workload being run."""
    for name in ("r02_traffic.json", "r01b_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(p):
            continue
        t = json.load(open(p))
        if t.get("workload") == workload and t.get("minibatch_per_gpu") == minibatch and kernel in t.get("kernels", {}):
            return t["kernels"][kernel]
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def workload_shape(cfg, actor, batch, dev, precision):
    """Rows the message-passing kernels actually process for one minibatch (after EMPN row pruning)."""
    from geometry_rl_b200.tensors import to_device
    policy = actor.get_submodule("0").module
    try:
        with torch.no_grad():
            graph, _ = policy.hyper_data.build_data(*[to_device(batch, dev)[k] for k in actor.in_keys], train=False)
        if cfg.model == "empn" and getattr(policy.gnn, "prune_dead_rows", False):
            pr = graph.homogeneous_pruned()
            n, e = pr.es.n_src, pr.es.n_edges
            rows = (f"EMPN rows that reach the readout only: {n} live of {graph.num_nodes} padded nodes, {e} edges; last layer at "
                    f"{pr.sub.n_dst} output nodes over {pr.sub.n_edges} edges (outputs and gradients identical to the dense "
                    f"evaluation, tests/test_gpu_parity.py::test_pruned_rows_equal_dense_evaluation)")
        elif cfg.model == "empn":
            es = graph.homogeneous()
            n, e, rows = es.n_src, es.n_edges, "dense (all padded nodes, every layer)"
        elif cfg.model == "hepi" and getattr(policy.gnn, "prune_dead_rows", False):
            pr = graph.hetero_pruned()
            n, e = pr.num_nodes, sum(es.n_edges for es in pr.edge_sets.values())
            rows = (f"HEPi rows that reach the readout only: {n} live of {graph.num_nodes} padded nodes, {e} edges (outputs and "
                    f"gradients identical to the dense evaluation)")
        else:
            n = graph.num_nodes
            e = sum(es.n_edges for es in graph.edge_sets.values())
            rows = "dense"
        return {"latent_mb": n * 4096 / 1e6, "basis_mb": e * (2048 if precision == "bf16" else 4096) / 1e6, "rows": rows}
    except Exception as exc:  # reporting only
        return {"latent_mb": float("nan"), "basis_mb": float("nan"), "rows": f"unavailable ({exc})"}


# algorithmic HBM bytes of ONE launch of each kernel: SURVEY 8(d)'s per-unit figures x the units the launch processes
# (R = 4096 B fp32 latent row, weights L2-resident and not counted, the edge basis recomputed on the fly and therefore
# worth ZERO bytes; 40 B per edge = two int64 indices + two positions as SURVEY counts them)
R = 16 * 64 * 4


def kernel_bytes(name, shape):
    n_src, n_dst, E = shape
    return {
        # fused 16-bit edge kernels (round 2): unique src rows read + x1 written / g_x1 read, x_src read, g_x_src written
        "grl_fbconv_edge_fused_fwd": n_src * R + n_dst * R + 40 * E,
        "grl_fbconv_edge_fused_bwd": 2 * n_src * R + n_dst * R + 40 * E,
        # node update: x1 read, x_dst read, out write (forward); grad_out read, x2 read, g_x1 write (backward).  The x2 row
        # the forward saves and the g_x2 round trip between the two backward kernels are implementation choices and are
        # NOT counted (they show up in `traffic`)
        "grl_fbconv_node_fwd_tc": 3 * n_dst * R,
        "grl_fbconv_node_bwd_tc": 3 * n_dst * R,
        "grl_fbconv_node_fwd": 3 * n_dst * R,
        "grl_fbconv_node_bwd": 3 * n_dst * R,
        "grl_absmax": n_dst * R,
        # round-1 kernels with a materialised basis (GRL_FUSED_EDGE=0 / strict fp32 path): by SURVEY 8(d) the basis rows are
        # not compulsory traffic, so they are not counted here either
        "grl_edge_basis_fwd": 40 * E, "grl_edge_basis_bwd": 40 * E,
        "grl_edge_basis_fwd_tc": 40 * E, "grl_edge_basis_bwd_tc": 40 * E,
        "grl_fbconv_edge_fwd": n_src * R + n_dst * R + 8 * E,
        "grl_fbconv_edge_fwd_tc": n_src * R + n_dst * R + 8 * E,
        "grl_fbconv_edge_bwd": 2 * n_src * R + n_dst * R + 12 * E,
        "grl_fbconv_edge_bwd_tc": 2 * n_src * R + n_dst * R + 12 * E,
    }.get(name)


def resolve_minibatch(args, cfg_name, cfg):
    return args.minibatch or DEFAULT_MINIBATCH.get(cfg_name, cfg.mini_batch_size)


def config_block(args, cfg_name, cfg, B, world):
    """The `config` object of the JSON line; identical for our arm and the reference arm (same workload, same sizes)."""
    return {"workload": cfg_name, "body": cfg.model, "minibatch_per_gpu": B, "global_minibatch": B * world,
            "parallelism": f"dp{world}",
            "inputs": f"{N_ROTATE} distinct synthetic minibatches (fixed seeds, independent of the kernels) rotated through "
                      f"the timed region; the per-step working set (hundreds of MB of latents) exceeds the 126 MB L2"}


def nominal_policy_output(cfg, B):
    """(mean, variance, value) the synthetic old distribution drifts from: the freshly initialised Gaussian head's output
    (mean 0, variance init_std**2 = 1: the initial policy's means are O(1e-2) and its variances within 2 % of 1) and a
    zero value, as the initial critic's values are O(1e-3).  Taken from the initialisation rather than from a forward
    pass, so that the minibatches do not depend on the kernels being measured."""
    k = cfg.total_action_dim
    return torch.zeros(B, k), torch.ones(B, k), torch.zeros(B, 1)


DUMP_MAX_BYTES = 64 << 20


def named_parameters(lrn, prefix):
    return {f"{prefix}.{net_name}.{k}": v for net_name, net in (("actor", lrn.actor), ("critic", lrn.critic))
            for k, v in net.named_parameters()}


def host_arrays(tensors):
    """Host copies keyed by `--dump-outputs` file names (float64 stays float64, everything else becomes float32)."""
    arrays = {}
    for k, v in tensors.items():
        v = v.detach().cpu()
        arrays[re.sub(r"[^A-Za-z0-9_.-]", "_", k)] = (v if v.dtype == torch.float64 else v.float()).numpy().copy()
    if len(arrays) != len(tensors):
        raise RuntimeError("--dump-outputs: two outputs map to the same file name")
    return arrays


def dump_outputs(path, arrays):
    """DIR/<name>.npy for every array.  Above DUMP_MAX_BYTES in all, every array keeps the same fraction of its elements:
    a fixed sample (flattened indices drawn by numpy.random.default_rng(0), in ascending order)."""
    budget = DUMP_MAX_BYTES - 128 * len(arrays)  # .npy headers
    frac = min(1.0, budget / sum(a.nbytes for a in arrays.values()))
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        if frac < 1.0:
            idx = np.sort(np.random.default_rng(0).choice(a.size, max(1, int(a.size * frac)), replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle port of the same step on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_step_rate(cfg, sample, steps, warmup, seed=0):
    from geometry_rl_b200 import learner
    from geometry_rl_b200.synthetic import synthetic_obs
    from oracle.step import OracleAgent, make_minibatch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    actor, critic, _, _, _ = learner.build_agent(cfg, "cpu", seed=seed)
    agent = OracleAgent(cfg, actor.state_dict(), critic.state_dict())
    gen = torch.Generator().manual_seed(1234)
    obs = synthetic_obs(cfg, sample, gen, env_ids=torch.arange(sample) * max(1, cfg.num_envs // sample) % cfg.num_envs)
    mb = make_minibatch(cfg, agent, obs, gen)
    params = [p for p in list(agent.actor.values()) + list(agent.critic.values()) if p.is_floating_point()]
    opt = torch.optim.Adam(params, lr=cfg.lr, eps=1e-5)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        agent.step_grads(mb)
        if cfg.clip_grad_norm:
            torch.nn.utils.clip_grad_norm_(params, cfg.max_grad_norm)
        opt.step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    return sample * len(times) / total, cores, total / len(times)


def run_reference(args):
    """The reference's own CPU implementation of the path, timed on the box's host cores with every thread torch can
    use.  The reference cannot be installed or imported here (torchrl / tensordict / PyG / ITPAL wheels are absent and
    /root/reference does not exist on the GPU box), so this is the CPU oracle port of the same step (kind = "port").
    Same workload, sizes, K and W as our arm; each step is a bounded sample (`--cpu-sample` graphs of the same synthetic
    minibatch) so that the run ends within a few minutes."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from geometry_rl_b200.synthetic import CONFIGS
    cfg = CONFIGS[args.config]
    B = resolve_minibatch(args, args.config, cfg)
    rate, cores, sec = cpu_step_rate(cfg, args.cpu_sample, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_block(args, args.config, cfg, B, world),
        "cpu_baseline": {"value": rate, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} update steps of {args.cpu_sample} graphs each after {args.warmup} warm-up steps "
                                   f"(a bounded sample of the {B}-graph minibatch; oracle/step.py = torch CPU fp32 restatement "
                                   f"of the reference step, fp64 KL dual solve instead of ITPAL)"},
        "e2e": {"value": rate, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(json.dumps(line))


def topology_rebuild_cost(dev, precision, name="rope_shaping_hepi_trpl_cfg", B=2048, steps=10):
    """BASELINE configs[3] extension: the rope policy graph's kNN topology rebuilt from the current link positions at
    every update (`hyper_data.rebuild_every_call`) against the reference's build-once rule, both launched eagerly (the
    rebuilt topology has host-visible sizes, so that mode cannot be replayed from a CUDA graph), plus the graph
    construction alone (kNN + dense task edges + dst/src CSR + live-row sets).  Single process; reporting only."""
    from geometry_rl_b200 import learner, ops
    from geometry_rl_b200.synthetic import CONFIGS, synthetic_minibatch, synthetic_obs
    from geometry_rl_b200.tensors import to_device
    ops.set_precision(precision)
    cfg = CONFIGS[name]
    actor, critic, _, loss_module, _ = learner.build_agent(cfg, dev, seed=0)
    lrn = learner.Learner(cfg, actor, critic, loss_module)
    gen = torch.Generator().manual_seed(4321)
    obs = synthetic_obs(cfg, B, gen, env_ids=torch.arange(B) % cfg.num_envs)
    lrn.calibrate(to_device(obs, dev))
    with torch.no_grad():
        d_ = actor.get_dist(to_device(obs, dev))
        v = critic.module(*[obs[k].to(dev) for k in critic.in_keys])
    mb = to_device(synthetic_minibatch(obs, d_.mean, d_.var_diag, v, gen), dev)
    hd = actor.module.hyper_data if hasattr(actor, "module") and hasattr(actor.module, "hyper_data") else None
    if hd is None:
        for m in actor.modules():
            if hasattr(m, "hyper_data"):
                hd = m.hyper_data
                break

    def timed(fn, n):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    out = {"workload": f"{name}@{B}", "launch": "eager (no CUDA graph)", "steps": steps}
    hd.rebuild_every_call = False
    out["build_once_ms_per_step"] = timed(lambda: lrn.update(mb), steps)
    hd.rebuild_every_call = True
    out["rebuild_every_step_ms_per_step"] = timed(lambda: lrn.update(mb), steps)
    pol_obs = [mb[k] for k in actor.in_keys] if hasattr(actor, "in_keys") else None

    def build_only():
        hd.invalidate()
        g, _ = hd.build_data(*pol_obs, train=True)
        if g.output_mask_key is not None:
            g.hetero_pruned()

    if pol_obs is not None:
        out["graph_construction_only_ms"] = timed(build_only, steps)
    hd.rebuild_every_call = False
    out["samples_per_s_rebuild"] = B / (out["rebuild_every_step_ms_per_step"] * 1e-3)
    out["samples_per_s_build_once"] = B / (out["build_once_ms_per_step"] * 1e-3)
    return out


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def measure(args, cfg_name, B, precision, dev, dp, rank, world, local, steps, full=True):
    """Build a fresh agent, capture the update, time `repeats` regions of exactly `steps` replayed updates with inputs
    resident in HBM (median region reported) and, with `full`, the end-to-end figure from pinned host memory plus the
    per-kernel CUDA-event pass.  Returns a dict of results (meaningful on rank 0)."""
    import torch.distributed as dist
    from geometry_rl_b200 import _lib, learner, ops
    from geometry_rl_b200.synthetic import CONFIGS, synthetic_minibatch, synthetic_obs
    from geometry_rl_b200.tensors import to_device

    # only the message-passing MLP contractions are 16-bit (north_star); the library GEMMs of the DeepSets critic and of
    # the Gaussian head stay fp32 (no TF32), so the critic branch keeps fp32 parity in both modes
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    ops.set_precision(precision)
    cfg = CONFIGS[cfg_name]
    actor, critic, projection, loss_module, adv_module = learner.build_agent(cfg, dev, seed=0)  # same init on all ranks
    lrn = learner.Learner(cfg, actor, critic, loss_module, dp=dp)

    dump = full and rank == 0 and args.dump_outputs
    # ---- synthetic minibatches of this rank's environments (weak scaling: B samples per GPU) -----------
    gen = torch.Generator().manual_seed(1234 + rank)
    host_batches = []
    for i in range(N_ROTATE):
        # slot j always belongs to the same env block -> the same geometry as the cached topology of slot j
        env_ids = (torch.arange(B) * max(1, cfg.num_envs // B) + rank) % cfg.num_envs
        obs = synthetic_obs(cfg, B, gen, env_ids=env_ids)
        if i == 0:
            lrn.calibrate(to_device(obs, dev))  # one-time kernel calibration (global statistics under DP)
            init = host_arrays(named_parameters(lrn, "init")) if dump else None
        mb = synthetic_minibatch(obs, *nominal_policy_output(cfg, B), gen)
        host_batches.append({k: t.pin_memory() for k, t in mb.items()})
    dev_batches = [to_device(b, dev) for b in host_batches]
    h2d_bytes = sum(t.numel() * t.element_size() for t in host_batches[0].values())

    def barrier():
        torch.cuda.synchronize()
        if dp is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if dp is None:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    # ---- device-resident timing ----------------------------------------------------------------------
    use_graph = not args.no_graph and (dp is None or not args.no_dp_graph)
    launches_per_step = None
    if use_graph:
        c0 = _lib.launch_count
        n_cap = max(args.warmup, 3)
        lrn.capture(dev_batches[0], warmup=n_cap)
        launches_per_step = (_lib.launch_count - c0) // (n_cap + 1)
        step = lrn.update_graphed
    else:
        step = lrn.update
    for i in range(args.warmup):
        step(dev_batches[i % N_ROTATE])
    repeats = args.repeats if full else min(args.repeats, 3)
    sampler = ClockSampler(list(range(world)) if world > 1 else local)
    barrier()
    if rank == 0 and full:
        sampler.start()
    launches0 = _lib.launch_count
    regions, host_ms = [], []
    torch.cuda.profiler.start()  # `ncu --profile-from-start off` captures exactly the timed steps
    for r in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        t_host = time.perf_counter()
        for i in range(steps):
            out = step(dev_batches[i % N_ROTATE])
        e1.record()
        host_ms.append((time.perf_counter() - t_host) * 1e3)  # host time to ENQUEUE the region (no sync inside)
        barrier()
        regions.append(max_over_ranks(e0.elapsed_time(e1)))
    torch.cuda.profiler.stop()
    # the later passes below run more updates: take the timed path's last outputs now
    outputs = None
    if dump:
        outputs = host_arrays({**{f"out.{k}": v for k, v in out.items() if torch.is_tensor(v)},
                               **{f"grad.{k}": v for k, v in lrn.flat_grads().items()}, **named_parameters(lrn, "param")})
        outputs.update(init)
    launches = launches_per_step * steps if use_graph else (_lib.launch_count - launches0) // repeats
    clocks = sampler.stop() if (rank == 0 and full) else None
    ms = sorted(regions)[len(regions) // 2]  # median K-step region (each region is exactly K steps, max over ranks)
    res = {"precision": precision, "value": B * world * steps / (ms * 1e-3), "ms_per_step": ms / steps, "steps": steps,
           "outputs": outputs,
           "clocks": clocks, "gpu_launches": launches, "cuda_graph": use_graph, "B": B, "model": cfg.model,
           "regions_ms": [round(x, 3) for x in regions],
           # host-side cost of enqueueing one step (max over ranks of the median region): close to ms_per_step means the
           # launching thread, not the GPU, paces the job
           "host_enqueue_ms_per_step": round(max_over_ranks(sorted(host_ms)[len(host_ms) // 2]) / steps, 3)}
    res.update(workload_shape(cfg, actor, host_batches[0], dev, precision))
    if not full:
        del lrn, actor, critic, loss_module, dev_batches, host_batches
        torch.cuda.empty_cache()
        return res

    # ---- optional device timeline of ONE step on rank 0 (GRL_TIMELINE=<path>; every rank runs the step: it holds
    # collectives).  Compact list of [name, stream, start_us, dur_us]; read with tools/timeline_summary.py. -----------
    tl_path = os.environ.get("GRL_TIMELINE")
    if tl_path:
        from torch.profiler import ProfilerActivity, profile
        barrier()
        # every rank records its own copy (rank r > 0 writes <path>.rank<r>): a straggler shows up as the rank whose
        # kernels are long, not as the rank that waits for it inside the gradient all-reduce
        my_path = tl_path if rank == 0 else f"{tl_path}.rank{rank}"
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step(dev_batches[0])
            torch.cuda.synchronize()
        trace = my_path + ".trace.json"
        prof.export_chrome_trace(trace)
        ev = json.load(open(trace)).get("traceEvents", [])
        rows = sorted(([e["name"], e.get("args", {}).get("stream"), e["ts"], e["dur"]] for e in ev
                       if e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset") and "ts" in e), key=lambda r: r[2])
        t0 = rows[0][2] if rows else 0
        json.dump([[r[0], r[1], round(r[2] - t0, 3), r[3]] for r in rows], open(my_path, "w"))
        os.remove(trace)
        barrier()

    # ---- end to end: pinned host minibatch -> H2D -> step -> loss scalar D2H, every step ----------------
    e2e_regions = []
    loss_host = 0.0
    for r in range(min(repeats, 5)):
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall = time.perf_counter()
        s0.record()
        if use_graph:
            lrn.prefetch(host_batches[0])
        for i in range(steps):
            if use_graph:
                # pinned host -> staging (H2D on a copy stream, issued one step ahead so it runs under the previous update)
                # -> the graph's static inputs (D2D) -> replay -> read the loss back.  Every step's inputs cross PCIe inside
                # the timed region; the copy of step i+1 overlaps the compute of step i.
                out = lrn.update_prefetched(host_batches[(i + 1) % N_ROTATE] if i + 1 < steps else None)
            else:
                out = step({k: t.to(dev, non_blocking=True) for k, t in host_batches[i % N_ROTATE].items()})
            loss_host = float(out["loss_trust_region"].item())  # device -> host read of the step's result
        s1.record()
        barrier()
        e2e_regions.append(max_over_ranks(max(s0.elapsed_time(s1), (time.perf_counter() - t_wall) * 1e3 if dp is None else 0.0)))
    e2e_ms = sorted(e2e_regions)[len(e2e_regions) // 2]
    res["e2e"] = {"value": B * world * steps / (e2e_ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": h2d_bytes,
                  "d2h_bytes_per_step": 4, "last_loss_trust_region": loss_host}

    # ---- per-kernel CUDA-event pass (same steps, eager, events around every C-ABI launch) -------------------
    res["roofline"] = None
    n_prof = min(steps, 5)
    if rank == 0:
        _lib.event_timing(True)
    for i in range(n_prof):  # every rank runs the steps (they contain collectives); only rank 0 records events
        lrn.update(dev_batches[i % N_ROTATE])
    torch.cuda.synchronize()
    if rank == 0:
        per_kernel = _lib.event_timing(False)  # name -> list of (ms, n_src, n_dst, n_edges)
        tot = {k: sum(x[0] for x in v) for k, v in per_kernel.items()}
        step_kernel_ms = sum(tot.values())
        top = max(tot, key=tot.get)
        peak, peak_src = measured_peaks()
        # average over the launches of the dominant kernel: algorithmic bytes of each launch / its duration
        ab = sum(kernel_bytes(top, x[1:]) or 0 for x in per_kernel[top])
        dur = tot[top] * 1e-3
        achieved = ab / dur / 1e9 if dur > 0 else 0.0
        fracs = {}
        for k, v in per_kernel.items():
            kb = sum(kernel_bytes(k, x[1:]) or 0 for x in v)
            if kb:
                fracs[k] = round(kb / (tot[k] * 1e-3) / 1e9 / peak, 4)
        res["roofline"] = {
            "bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": measured_traffic(top, cfg_name, B), "peak_source": peak_src,
            "accounting": "SURVEY 8(d): unique latent rows in/out + 40 B per edge; the recomputed edge basis counts zero bytes",
            "avg_launch_ms": tot[top] / len(per_kernel[top]), "launches_per_step": len(per_kernel[top]) / n_prof,
            "algorithmic_bytes_per_launch": ab / len(per_kernel[top]), "share_of_kernel_time": tot[top] / step_kernel_ms,
            "kernel_ms_per_step": {k: round(v / n_prof, 4) for k, v in sorted(tot.items(), key=lambda kv: -kv[1])},
            "frac_by_kernel": fracs}
    del lrn, actor, critic, loss_module, dev_batches, host_batches
    torch.cuda.empty_cache()
    return res


def gae_rate(dev, B, T, iters=50):
    """grl_gae_scan alone through the C ABI on pre-converted inputs (SURVEY 8(d): 'GAE reported separately'), at a size
    whose 18 B per frame exceed the L2: frames/s and achieved GB/s against the measured HBM peak."""
    import ctypes as C  # noqa: F401
    from geometry_rl_b200 import _lib as L
    g = torch.Generator().manual_seed(3)
    r, v = torch.randn(B, T, generator=g).to(dev), torch.randn(B, T + 1, generator=g).to(dev)
    done = torch.zeros(B, T, dtype=torch.uint8, device=dev)
    done[:, -1] = 1
    adv, vt = torch.empty_like(r), torch.empty_like(r)

    def call():
        L.call("grl_gae_scan", L.ptr(r), L.ptr(v), L.ptr(done), L.ptr(done), 0.99, 0.95, B, T, L.ptr(adv), L.ptr(vt))
    for _ in range(3):
        call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        call()
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) * 1e-3 / iters
    peak, _ = measured_peaks()
    gbs = 18 * B * T / sec / 1e9
    return {"frames_per_s": B * T / sec, "B_env": B, "T": T, "us_per_call": sec * 1e6, "GBps_at_18B_per_frame": gbs,
            "frac_of_hbm_peak": gbs / peak,
            "note": "kernel alone (one warp per env, Kogge-Stone scan of affine maps along T); 18 B per frame = 151 MB per call"}


def run_ours(args):
    import torch.distributed as dist
    from geometry_rl_b200 import _lib
    from geometry_rl_b200.synthetic import CONFIGS

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.load()
    dp = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        from geometry_rl_b200.parallel import DataParallel
        dp = DataParallel(side_group=not args.no_dp_overlap)
    cfg = CONFIGS[args.config]
    B = resolve_minibatch(args, args.config, cfg)

    main_res = measure(args, args.config, B, args.precision, dev, dp, rank, world, local, args.steps)
    if main_res["outputs"] is not None:
        dump_outputs(args.dump_outputs, main_res["outputs"])
    # the other precision mode of the same path, measured in the same run (one region; no per-kernel pass)
    other = "fp32" if args.precision == "bf16" else "bf16"
    other_res = None
    if not args.single_precision and cfg.model != "transformer":
        other_res = measure(args, args.config, B, other, dev, dp, rank, world, local, min(args.steps, 5), full=False)
    side = {}
    if not args.no_side_workloads:
        for name, b in SIDE_WORKLOADS:
            if (name, b) == (args.config, B):
                continue
            try:
                r = measure(args, name, b, args.precision, dev, dp, rank, world, local, args.steps, full=False)
                side[f"{name}@{b}"] = {"value": r["value"], "unit": "samples/s", "ms_per_step": r["ms_per_step"],
                                       "minibatch_per_gpu": b, "global_minibatch": b * world, "steps": r["steps"],
                                       "regions_ms": r["regions_ms"], "rows": r["rows"]}
            except Exception as exc:  # a side workload must not take the headline down
                side[f"{name}@{b}"] = {"error": f"{type(exc).__name__}: {exc}"}

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        rate, cores, sec = cpu_step_rate(cfg, args.cpu_sample, 3, 1)
        cpu = {"value": rate, "unit": "samples/s", "cores": cores, "kind": "port",
               "sample": f"3 update steps of {args.cpu_sample} graphs after 1 warm-up (a bounded sample of the {B}-graph minibatch; "
                         f"oracle/step.py: torch CPU fp32 restatement of the reference step, fp64 KL dual solve instead of "
                         f"ITPAL), {sec:.2f} s/step"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": main_res["value"], "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic",
            "config": config_block(args, args.config, cfg, B, world),
            "details": {"mlp_precision": args.precision,
                        "parity": "1e-5 vs reference fp32" if args.precision == "fp32" else
                                  "1e-2 vs reference fp32 (north_star 16-bit MLP path: tcgen05 operands in fp16 / bf16, fp32 "
                                  "accumulation; latents, LayerNorm, segmented sums, projection, losses fp32; "
                                  "tests/test_gpu_step16.py)",
                        "cuda_graph": main_res["cuda_graph"], "rows": main_res["rows"],
                        "timing": f"{len(main_res['regions_ms'])} timed regions of exactly {args.steps} steps each (barrier + "
                                  f"synchronize on both sides, CUDA events, max over ranks); value = median region",
                        "regions_ms": main_res["regions_ms"],
                        "host_enqueue_ms_per_step": main_res["host_enqueue_ms_per_step"],
                        "latent_mb": main_res["latent_mb"]},
            "clocks": main_res["clocks"], "e2e": main_res["e2e"], "gpu_launches": main_res["gpu_launches"],
            "roofline": main_res["roofline"], "cpu_baseline": cpu, "configs": side,
        }
        if not args.no_side_workloads and dp is None:
            try:
                line["topology_rebuild"] = topology_rebuild_cost(dev, args.precision)
            except Exception as exc:  # reporting only
                line["topology_rebuild"] = {"error": f"{type(exc).__name__}: {exc}"}
        try:
            line["gae"] = gae_rate(dev, 65536, 128)
        except Exception as exc:  # reporting only
            line["gae"] = {"error": str(exc)}
        if other_res is not None:
            line["other_precision"] = {"mlp_precision": other, "dtype": "f32" if other == "fp32" else "bf16",
                                       "value": other_res["value"], "unit": "samples/s", "ms_per_step": other_res["ms_per_step"],
                                       "steps": other_res["steps"],
                                       "parity": "1e-5 vs reference fp32" if other == "fp32" else "1e-2 vs reference fp32"}
        _emit(json.dumps(line))
    if dp is not None:
        dist.destroy_process_group()


def main():
    args = parse()
    # the contract is ONE JSON line on stdout: library chatter goes to stderr — at the file-descriptor level too, because
    # NCCL prints its version banner with C stdio ("NCCL version 2.28.9+cuda12.9")
    sys.stdout.flush()
    real_fd = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    global _emit
    _emit = lambda line: os.write(real_fd, (line + "\n").encode())
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
