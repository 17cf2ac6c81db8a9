"""Observation normalisation of the collection side (SURVEY 8(f) N4): `ReshapeTransform` and `NDVecNorm` with the
reference's class names and keyword arguments (geometry_rl/torchrl/envs/transforms.py:72-171), as plain callables on
any mapping of tensors (a TensorDict included) — torchrl / tensordict are not installable offline.

What the reference does with them (configs/rigid_insertion_multi_hepi_trpl_cfg.yaml:46-58): the flat
`position_vectors` / `velocity_vectors` groups are reshaped to [B_env, n, 3] and standardised per xyz COMPONENT
(`shapes: [3, 3]`): the running statistics have shape [3] and are shared by every point of every environment; the
results are written to `norm_position_vectors` / `norm_velocity_vectors`.  These are the `norm_*` inputs of the graph
feature builder (pyg_data/*_tasks_data.py).

[3P-memory] PARITY UNPINNED: `NDVecNorm` only overrides `_call` (it passes N = product of ALL leading dimensions to
`_update` instead of the tensordict batch size, transforms.py:147-151); the arithmetic lives in torchrl 0.3.1's
`VecNorm._update`, restated here from the pinned version:
    sum  <- decay * sum  + sum_over_leading_dims(x)        ssq <- decay * ssq + sum_over_leading_dims(x^2)
    count <- decay * count + N
    mean = sum / count;  std = sqrt(clamp_min(ssq / count - mean^2, eps));  out = (x - mean) / clamp_min(std, eps)
The statistics update BEFORE the value is standardised (the current batch is part of its own statistics).
Everything stays on the tensor's device; the three reductions are torch sums (deterministic)."""
from typing import Dict, List, Mapping, MutableMapping, Optional, Sequence

import torch


class ReshapeTransform:
    """transforms.py:72-132: `obs.reshape([obs.shape[0]] + out_shape)` for every in_key (batch dimension kept)."""

    def __init__(self, in_keys: Optional[Sequence[str]] = None, out_keys: Optional[Sequence[str]] = None, *,
                 out_shape: Optional[Sequence[int]] = None, **ignored):
        if out_shape is None:
            raise ValueError("shape must be specified")
        self.in_keys = list(in_keys or [])
        self.out_keys = list(out_keys) if out_keys is not None else list(self.in_keys)
        self.out_shape = list(out_shape)
        self._original_shape = None

    def __call__(self, td: MutableMapping[str, torch.Tensor]):
        for k, ok in zip(self.in_keys, self.out_keys):
            if k in td:
                obs = td[k]
                self._original_shape = obs.shape
                td[ok] = obs.reshape([obs.shape[0]] + self.out_shape)
        return td

    def inv(self, state: torch.Tensor) -> torch.Tensor:
        return state.reshape(self._original_shape)


class NDVecNorm:
    """transforms.py:135-171 on top of torchrl 0.3.1 `VecNorm(in_keys, out_keys, shapes, decay, eps)`.

    `shapes[i]` is the TRAILING shape the statistics of in_keys[i] are kept in ([3]: one mean / std per xyz component);
    every leading dimension (environments, points) is summed over and counted (`_count_left`, transforms.py:62-68)."""

    def __init__(self, in_keys: Sequence[str], out_keys: Optional[Sequence[str]] = None, shapes: Optional[Sequence] = None,
                 decay: float = 0.9999, eps: float = 1e-4, *, dp=None, **ignored):
        """`dp`: a `parallel.DataParallel` handle; `apply_device` then takes its statistics over every rank's rows."""
        self.in_keys = list(in_keys)
        self.dp = dp
        self.out_keys = list(out_keys) if out_keys is not None else list(self.in_keys)
        if shapes is not None and len(shapes) != len(self.in_keys):
            raise ValueError("shapes must have one entry per in_key")
        self.shapes = [tuple([s] if isinstance(s, int) else s) for s in shapes] if shapes is not None else None
        self.decay, self.eps = float(decay), float(eps)
        self.frozen = False
        self._stats: Dict[str, Dict[str, torch.Tensor]] = {}

    def _init(self, key: str, value: torch.Tensor):
        if key in self._stats:
            return
        i = self.in_keys.index(key)
        shape = self.shapes[i] if self.shapes is not None else tuple(value.shape[1:])
        if tuple(value.shape[value.dim() - len(shape):]) != tuple(shape):
            raise ValueError(f"{key}: trailing shape {tuple(value.shape)} does not end in {tuple(shape)}")
        z = lambda: torch.zeros(shape, dtype=value.dtype, device=value.device)
        self._stats[key] = {"sum": z(), "ssq": z(), "count": torch.zeros(1, dtype=value.dtype, device=value.device)}

    @torch.no_grad()
    def _update(self, key: str, value: torch.Tensor) -> torch.Tensor:
        st = self._stats[key]
        lead = tuple(range(value.dim() - st["sum"].dim()))
        n = 1
        for d in lead:
            n *= value.shape[d]
        if not self.frozen:
            st["sum"].mul_(self.decay).add_(value.sum(lead) if lead else value)
            st["ssq"].mul_(self.decay).add_(value.pow(2).sum(lead) if lead else value.pow(2))
            st["count"].mul_(self.decay).add_(max(1, n))
        mean = st["sum"] / st["count"]
        std = (st["ssq"] / st["count"] - mean.pow(2)).clamp_min(self.eps).sqrt()
        return (value - mean) / std.clamp_min(self.eps)

    def __call__(self, td: MutableMapping[str, torch.Tensor]):
        for k, ok in zip(self.in_keys, self.out_keys):
            if k not in td:
                continue
            v = td[k]
            self._init(k, v)
            td[ok] = self._update(k, v)
        return td

    # ---- what train.py:343-365 checkpoints of the transform -------------------------------------------------------
    def state_dict(self) -> Dict[str, torch.Tensor]:
        return {f"{k}_{n}": t.clone() for k, st in self._stats.items() for n, t in st.items()}

    def load_state_dict(self, sd: Mapping[str, torch.Tensor]):
        """Copies into the existing state tensors when they have the checkpoint's shapes (a CUDA graph captured with
        `PolicyOperator.capture_act(obs_norm=...)` keeps reading them), else installs clones."""
        for k in self.in_keys:
            if f"{k}_sum" in sd:
                new = {n: sd[f"{k}_{n}"] for n in ("sum", "ssq", "count")}
                st = self._stats.get(k)
                if st is not None and all(st[n].shape == new[n].shape and st[n].dtype == new[n].dtype for n in new):
                    for n, t in new.items():
                        st[n].copy_(t)
                else:
                    self._stats[k] = {n: t.clone() for n, t in new.items()}

    def freeze(self):
        """Evaluation mode (`VecNorm.freeze()`): standardise with the current statistics without updating them."""
        self.frozen = True
        return self

    # ---- the device path (csrc/grl_obsnorm.cu) ---------------------------------------------------------------------
    def ensure_stats(self, td: Mapping[str, torch.Tensor]):
        """Create (zeros) or move the statistics of every present in_key to its tensor's device, as fp32 contiguous
        tensors.  `apply_device` does this itself; a CUDA graph capture calls it first so that no allocation or memset of
        the state is recorded."""
        for i, k in enumerate(self.in_keys):
            if k not in td:
                continue
            v = td[k]
            shape = self.shapes[i] if self.shapes is not None else tuple(v.shape[1:])
            st = self._stats.get(k)
            if st is None:
                z = lambda: torch.zeros(shape, dtype=torch.float32, device=v.device)
                self._stats[k] = {"sum": z(), "ssq": z(), "count": torch.zeros(1, dtype=torch.float32, device=v.device)}
            elif any(t.device != v.device or t.dtype != torch.float32 or not t.is_contiguous() for t in st.values()):
                self._stats[k] = {n: t.to(device=v.device, dtype=torch.float32).contiguous() for n, t in st.items()}
        return self

    @torch.no_grad()
    def apply_device(self, td: MutableMapping[str, torch.Tensor], out: Optional[Mapping[str, torch.Tensor]] = None):
        """What `__call__` computes, on the device kernels (`ops.vecnorm`), for every present in_key at once, on the same
        state tensors.  The input keeps its layout: a flat [B, F] group is read as B F / C rows of the C statistics
        components (ReshapeTransform is a view), and td[out_key] has x's shape.  `out` (out_key -> tensor) names the
        output tensors; otherwise new ones are allocated.  With `dp` the increments are summed over all ranks (equal
        shards) before the update, so every rank holds bit-identical statistics."""
        from ...ops import vecnorm
        keys = [(k, ok) for k, ok in zip(self.in_keys, self.out_keys) if k in td]
        if not keys:
            return td
        self.ensure_stats(td)
        xs = [td[k] for k, _ in keys]
        outs = [out[ok] if out is not None else torch.empty_like(x) for (_, ok), x in zip(keys, xs)]
        st = [self._stats[k] for k, _ in keys]
        vecnorm(xs, out=outs, sums=[s["sum"] for s in st], ssqs=[s["ssq"] for s in st], counts=[s["count"] for s in st],
                decay=self.decay, eps=self.eps, update=not self.frozen,
                all_reduce=self.dp.all_reduce if self.dp is not None else None,
                world_size=self.dp.world_size if self.dp is not None else 1)
        for (_, ok), o in zip(keys, outs):
            td[ok] = o
        return td
