"""Data parallelism over minibatch samples (one process per GPU, torch.distributed; NCCL on the box, gloo
in CPU tests).  The reference is single-process (SURVEY 2.1); to stay results-equivalent to it, every
cross-sample reduction of the update step is made global here (SURVEY 8(e)):

  * advantage mean / unbiased std                       (objectives/trpl.py:286-289)
  * loss means (local sum / global count) + ONE summed gradient bucket per network
  * PyG LayerNorm(mode='graph') statistics of the DeepSets critic, forward and backward
  * ESS logsumexp and the logged metric means / maxima  (trpl.py:294-300, base_projection_layer.py:355-369)

Equal shard sizes are required (every rank holds B_global / world_size samples)."""
from typing import Dict, Iterable, List

import torch
import torch.distributed as dist


class _GraphNormStats(torch.autograd.Function):
    """(mean, biased std) of the GLOBAL tensor per group from local rows; gradients flow back to local rows."""

    @staticmethod
    def forward(ctx, xg, dp):
        n_local = xg.shape[1]
        s = torch.stack([xg.sum(1), (xg * xg).sum(1)], 0)  # [2, G]
        dp.all_reduce(s)
        n = n_local * dp.world_size
        mean = s[0] / n
        var = (s[1] / n - mean * mean).clamp_min(0)
        std = var.sqrt()
        ctx.save_for_backward(xg, mean, std)
        ctx.dp, ctx.n = dp, n
        return mean[:, None], std[:, None]

    @staticmethod
    def backward(ctx, g_mean, g_std):
        xg, mean, std = ctx.saved_tensors
        g = torch.stack([g_mean[:, 0], g_std[:, 0]], 0).contiguous()
        ctx.dp.all_reduce(g)  # every rank's loss depends on the shared statistics
        gm, gs = g[0][:, None], g[1][:, None]
        gx = gm / ctx.n + gs * (xg - mean[:, None]) / (ctx.n * std[:, None])
        return gx, None


SIDE_STREAM_RESERVED_SMS = 4

_split_capture = None  # set while a SegmentedGraph records: DataParallel.all_reduce then ends the current segment


class SegmentedGraph:
    """A CUDA graph split at every `DataParallel.all_reduce` the captured function issues.  Each collective runs between
    the replays of two segments, on the static tensor the first one wrote, so the replay works with any backend (gloo
    cannot be captured, and ranks that share one GPU cannot use NCCL).  The segments share one memory pool and always
    replay in capture order.  A function without collectives gives one segment: a plain CUDA graph."""

    def capture(self, fn):
        global _split_capture
        pool = torch.cuda.graph_pool_handle()
        parts, cur = [], [None]

        def begin():
            g = torch.cuda.CUDAGraph()
            g.capture_begin(pool=pool)
            cur[0] = g

        def split(dp, t, op):
            cur[0].capture_end()
            parts.append((cur[0], dp, t, op))
            begin()

        torch.cuda.synchronize()
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(stream):
            begin()
            _split_capture = split
            try:
                out = fn()
            finally:
                _split_capture = None
                cur[0].capture_end()
        torch.cuda.current_stream().wait_stream(stream)
        self.parts, self.last = parts, cur[0]
        return out

    def replay(self):
        for g, dp, t, op in self.parts:
            g.replay()
            dp.all_reduce(t, op)
        self.last.replay()


class DataParallel:
    def __init__(self, group=None, side_group: bool = False):
        """`side_group=True` creates a SECOND communicator (`self.side`) for the critic branch: the learner then
        runs that branch on its own CUDA stream under the actor's kernels, and its graph-LayerNorm statistics
        all-reduce on `side` while the actor-side reductions and the gradient bucket use the main communicator
        (collectives of one communicator must stay ordered; two streams need two communicators)."""
        if not dist.is_initialized():
            raise RuntimeError("torch.distributed is not initialised")
        self.group = group
        self.world_size = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.collectives = 0
        self.side = DataParallel(group=dist.new_group(), side_group=False) if side_group else None
        if side_group and torch.cuda.is_available():
            # The critic branch's collectives then run CONCURRENTLY with the actor's persistent kernels.  A collective
            # that waits for a late rank spins on its SMs, and a persistent grid that fills every SM cannot place the CTAs
            # that belong there until it ends: measured at 8 GPUs (profiles/r02_timeline_n8_ranks.md) the edge backward
            # stretched from 1.8 to 3.3 ms under a 1.7 ms all-reduce, on most ranks.  Tiny collectives use one CTA each;
            # two communicators can be active at once: four SMs stay out of the kernels' grids.
            from . import _lib
            _lib.reserve_sms(SIDE_STREAM_RESERVED_SMS)

    def all_reduce(self, t: torch.Tensor, op=dist.ReduceOp.SUM) -> torch.Tensor:
        if _split_capture is not None:  # recorded by a SegmentedGraph: the collective runs between its segments
            _split_capture(self, t, op)
            return t
        dist.all_reduce(t, op=op, group=self.group)
        self.collectives += 1
        return t

    def all_gather_small(self, t: torch.Tensor) -> torch.Tensor:
        """[n] -> [world, n] (ops.trpl_loss hook: one collective per loss stage, combined in rank order on the device)."""
        out = torch.empty(self.world_size * t.numel(), dtype=t.dtype, device=t.device)  # concatenated layout (gloo wants it flat)
        dist.all_gather_into_tensor(out, t.contiguous().reshape(-1), group=self.group)
        self.collectives += 1
        return out.view((self.world_size,) + tuple(t.shape))

    def all_reduce_named(self, t: torch.Tensor, op: str) -> torch.Tensor:
        """In-place all-reduce of a (view of a) small statistics tensor; `op` = "sum" | "max" (ops.trpl_loss hook)."""
        return self.all_reduce(t, dist.ReduceOp.SUM if op == "sum" else dist.ReduceOp.MAX)

    # ---- forward-side statistics ---------------------------------------------------------------------
    def mean_std_unbiased(self, x: torch.Tensor):
        x = x.detach().float()
        s = torch.stack([x.sum(), (x * x).sum()])
        self.all_reduce(s)
        n = x.numel() * self.world_size
        mean = s[0] / n
        var = (s[1] - n * mean * mean) / (n - 1)
        return mean, var.clamp_min(0).sqrt()

    def logsumexp(self, x: torch.Tensor) -> torch.Tensor:
        m = self.all_reduce(x.max().clone(), dist.ReduceOp.MAX)
        s = self.all_reduce((x - m).exp().sum())
        return m + s.log()

    def graph_norm_stats(self, xg: torch.Tensor):
        return _GraphNormStats.apply(xg, self)

    def aggregate_metrics(self, per_sample: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        keys = list(per_sample.keys())
        sums = torch.stack([per_sample[k].sum() for k in keys])
        maxs = torch.stack([per_sample[k].max() for k in keys])
        self.all_reduce(sums)
        self.all_reduce(maxs, dist.ReduceOp.MAX)
        n = per_sample[keys[0]].numel() * self.world_size
        out = {}
        for i, k in enumerate(keys):
            out[k] = sums[i] / n
            out[f"{k}_max"] = maxs[i]
        return out

    def global_losses(self, out: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """Logging view of a sharded TRPLLoss output: every `loss_*` entry is this rank's share (local sum / global
        count, so that summed gradients are the global-mean gradients); their sum over ranks is the reference's value."""
        keys = [k for k in out if k.startswith("loss_") or k == "actor_loss"]
        t = torch.stack([out[k].detach() for k in keys])
        self.all_reduce(t)
        res = dict(out)
        for i, k in enumerate(keys):
            res[k] = t[i]
        return res

    # ---- replica consistency ---------------------------------------------------------------------------
    def sync_module_state(self, *modules):
        """Broadcast every parameter and buffer from rank 0 (construction time).  Afterwards replicas only stay identical
        if every state change is a function of GLOBAL quantities: gradients are all-reduced, and the one-time kernel
        calibration of FiberBundleConv (conv.py:151-157) takes its std() over all ranks' rows (`global_std`)."""
        for m in modules:
            for t in list(m.parameters()) + list(m.buffers()):
                dist.broadcast(t.data, 0, group=self.group)

    def global_std(self, x: torch.Tensor) -> torch.Tensor:
        """Unbiased std of the concatenation of every rank's `x` (torch.Tensor.std() semantics) from fp64 moments."""
        x = x.detach().double()
        s = torch.stack([x.sum(), (x * x).sum(), torch.tensor(float(x.numel()), dtype=torch.float64, device=x.device)])
        self.all_reduce(s)
        n = s[2]
        var = (s[1] - s[0] * s[0] / n) / (n - 1)
        return var.clamp_min(0).sqrt().float()

    # ---- gradient exchange -----------------------------------------------------------------------------
    def allreduce_grads(self, params: Iterable[torch.nn.Parameter]):
        """ONE flat fp32 bucket, summed (losses already divide by the global count)."""
        ps: List[torch.nn.Parameter] = [p for p in params if p.requires_grad]
        for p in ps:
            if p.grad is None:  # e.g. the AGENT conv when A == 1: keep the bucket layout identical on all ranks
                p.grad = torch.zeros_like(p)
        flat = torch.cat([p.grad.reshape(-1) for p in ps])
        self.all_reduce(flat)
        off = 0
        for p in ps:
            n = p.numel()
            p.grad.copy_(flat[off:off + n].view_as(p))
            off += n
        return flat.numel()

    def attach(self, loss_module):
        """Install the global-statistics hooks on a TRPLLoss and on every GraphLayerNorm of its critic."""
        from .modules.pyg_models.pyg_compat import GraphLayerNorm
        from . import ops
        loss_module.dp = self
        actor = getattr(loss_module, "actor_network", None)
        if actor is not None:
            actor.act_rank = self.rank  # rollout noise (PolicyOperator.act*): the rank enters the key, one stream per rank
        ops.set_calibration_std(self.global_std)  # conv.py:151-157 / ponita.py:178-192 statistics become global
        critic_dp = self.side if self.side is not None else self
        for m in loss_module.critic_network.modules():
            if isinstance(m, GraphLayerNorm):
                m.stats_reduce = critic_dp.graph_norm_stats
                m.fused_all_reduce = (critic_dp.all_reduce, critic_dp.world_size)
        return loss_module
