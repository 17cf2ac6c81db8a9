"""Observation tensors -> batched graph + per-node features, on the GPU.

Mirrors the interface of the reference's `BaseData` (geometry_rl/modules/pyg_data/base_data.py:9-75):
`build_data(*obs_tensors, train=) -> (graph, input_vector)` with a topology cache keyed on the batch
size (`_should_reconstruct_placeholders`, rigid_tasks_data.py:254-255).  Differences in mechanism,
not in results:
  * topology is built by the batched K1 CUDA kernels instead of a Python loop of per-graph
    knn_graph calls; the coalesced COO it yields is bit-identical to the reference's edge_index;
  * `HeteroCartesian` / `HeteroDistance` edge attributes (recomputed every call by the reference,
    rigid_tasks_data.py:250, but read by none of HEPi / EMPN / DeepSets / transformer) are not produced.
"""
import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from ... import ops
from ..._lib import MAX_KNN as MAX_NUM_NEIGHBORS
from .graph import GraphBatch


def noise_like(tensor: torch.Tensor, std: float = 0.1) -> torch.Tensor:
    """pyg_data/utils.py:13-15."""
    return torch.randn_like(tensor) * std


class BaseData:
    # subclasses fill these in
    TASK: str = ""
    ALL_NODE_TYPES: Sequence[str] = ()
    PARTICLE_TYPE: str = ""
    ACTUATOR_TYPE: str = "grippers"
    INTERNAL_MODE: str = "knn"
    EDGE_TYPES: Sequence[Tuple[str, str, str]] = ()
    HAS_INFOS: bool = False
    HAS_NUM_VALID: bool = False  # the particle count varies per sample (`_num_valid`): kNN edge counts are data-dependent

    def __init__(self, observation_dim: Dict, observation_names: Dict, full_graph_obs: bool = False,
                 dist_as_pos: bool = False, output_mask_key: Optional[str] = None, training_noise: bool = False,
                 training_noise_std: float = 1e-2, concat_input_vector: bool = True, angular_velocity: bool = True,
                 knn_k: int = 3, knn_to_actuators_k: int = -1, build_edges: bool = True, internal_edges: str = "knn",
                 radius: Optional[float] = None, max_num_neighbors: int = MAX_NUM_NEIGHBORS, **kwargs):
        self._output_mask_key = output_mask_key
        self.training_noise = training_noise
        self.training_noise_std = training_noise_std
        self.concat_input_vector = concat_input_vector
        self.observation_dim = {k: [v[0] if isinstance(v, (tuple, list)) else int(v) for v in vs]
                                for k, vs in observation_dim.items()}
        self.observation_names = observation_names
        self.full_graph_obs = full_graph_obs
        self.dist_as_pos = dist_as_pos
        self.angular_velocity = angular_velocity
        self.knn_k = knn_k
        self.knn_to_actuators_k = knn_to_actuators_k
        # False for consumers that never read edges (DeepSets critic, transformer tokens): skips the K1 kernels
        self.build_edges = build_edges
        if knn_to_actuators_k > 0:
            # the reference's own kNN-to-actuator branch never assigns TASK edges for rigid tasks
            # (rigid_tasks_data.py:302-312) and no shipped config selects it
            raise NotImplementedError("knn_to_actuators_k > 0 is not reachable with the shipped configs")
        # INTERNAL edges of the kNN tasks (rigid, rope): "knn" (the reference's knn_graph, k = knn_k) or "radius" (every
        # point within `radius`, at most the `max_num_neighbors` nearest; ops.radius_graph).  Cloth's are "full".
        if internal_edges not in ("knn", "radius"):
            raise ValueError(f"internal_edges must be 'knn' or 'radius', not {internal_edges!r}")
        if internal_edges == "radius":
            if self.INTERNAL_MODE != "knn":
                raise ValueError(f"{type(self).__name__}: INTERNAL edges are '{self.INTERNAL_MODE}'; internal_edges="
                                 "'radius' applies to the kNN tasks (rigid, rope)")
            if isinstance(radius, bool) or not isinstance(radius, (int, float)) or not math.isfinite(radius) or radius <= 0:
                raise ValueError(f"internal_edges='radius' needs a finite radius > 0, got {radius!r}")
            if (isinstance(max_num_neighbors, bool) or not isinstance(max_num_neighbors, int)
                    or not 1 <= max_num_neighbors <= MAX_NUM_NEIGHBORS):
                raise ValueError(f"max_num_neighbors must be an int in [1, {MAX_NUM_NEIGHBORS}], got {max_num_neighbors!r}")
        elif radius is not None:
            raise ValueError("radius is only used with internal_edges='radius'")
        self.internal_edges = internal_edges
        self.radius = None if radius is None else float(radius)
        self.max_num_neighbors = max_num_neighbors
        self.node_type_list = self._kept_node_types()
        # The reference keeps ONE placeholder and rebuilds it whenever the incoming batch size differs from the last one
        # (rigid_tasks_data.py:254-255), i.e. at every rollout <-> minibatch size alternation.  Same rule here: the dict
        # holds a single entry unless `cache_all_sizes` is switched on (then the caller owns staleness: `invalidate()` at
        # every rollout -> update boundary restores the reference's refresh points).  A captured CUDA graph
        # (Learner.capture) holds the topology tensors it was recorded with: re-capture after an invalidation.
        self.cache_all_sizes = False
        # Extension (BASELINE configs[3], SURVEY 3.4): rebuild the kNN / task topology from the CURRENT positions on every
        # `build_data` call instead of re-using the placeholder of the first batch (rope_tasks_data.py:224-225,251 builds
        # once).  Off by default - parity runs use the reference's build-once rule.  Two ways (see `refresh_in_place`):
        #   * in place: radius INTERNAL edges consumed by the fused 16-bit path, or kNN INTERNAL edges with `knn_in_place`
        #     - the placeholder of the batch size is kept and its position- / num_valid-dependent edge types are rewritten
        #     on the device, no host sync, so a captured CUDA graph (Learner.capture, capture_act) rebuilds the topology on
        #     every replay;
        #   * eagerly (any other combination): the placeholder is dropped and rebuilt at exact size, with host syncs - not
        #     capturable.
        self.rebuild_every_call = False
        # Opt-in, with rebuild_every_call: rebuild kNN INTERNAL edges in place (ops.refresh_knn_edge_set).  Without
        # num_valid (rope) the set stays exact-size, so every precision and edge path consumes it; with num_valid (rigid)
        # it has a fixed capacity and needs the fused 16-bit path.  As with radius edges, pruning then keeps every row of
        # the node type and an edge type without edges still runs its convolution; the eager rebuild recomputes the
        # live rows per topology and skips such an edge type, as the reference does.
        self.knn_in_place = False
        # set by the policy wrapper: True when the model consumes fixed-capacity edge sets (HEPi)
        self.consumer_accepts_capacity = False
        # set by the policy wrapper: True when the model reads only the homogeneous views of GraphBatch (EMPN), which are
        # then merged on the device from fixed-capacity edge sets and refreshed with them
        self.consumer_accepts_homogeneous_capacity = False
        self._placeholders: Dict[int, GraphBatch] = {}
        self._example_data: Optional[GraphBatch] = None

    # ---- configuration hooks ---------------------------------------------------------------------
    def _kept_node_types(self) -> List[str]:
        raise NotImplementedError

    @property
    def example_data(self):
        return self._example_data

    def output_mask(self, data: GraphBatch, key: Optional[str]) -> slice:
        if key is not None:
            start = data.node_offsets[key]
            return slice(start, start + data.nodes_per_graph[key])
        return slice(None)

    # ---- public entry point (base_data.py:45-55) ----------------------------------------------------
    def refresh_in_place(self) -> bool:
        """True when `rebuild_every_call` rewrites the topology in place on the device (capturable): edges built, a model
        that accepts refreshed edge sets (HEPi), and either radius INTERNAL edges on the fused 16-bit edge path or kNN
        INTERNAL edges with `knn_in_place`, exact-size without num_valid, on the fused 16-bit path with it.  A model that
        reads the homogeneous view (EMPN) needs kNN INTERNAL edges with `knn_in_place` on the fused 16-bit path."""
        if not (self.rebuild_every_call and self.build_edges):
            return False
        if self.consumer_accepts_homogeneous_capacity and not self.consumer_accepts_capacity:
            return (self.knn_in_place and self.internal_edges == "knn" and self.INTERNAL_MODE == "knn"
                    and ops.fused_edge_enabled())
        if not self.consumer_accepts_capacity:
            return False
        if self.internal_edges == "radius":
            return ops.fused_edge_enabled()
        return (self.knn_in_place and self.INTERNAL_MODE == "knn"
                and (not self.HAS_NUM_VALID or ops.fused_edge_enabled()))

    def build_data(self, *args, **kwargs):
        inputs = self._preprocess_input(*args, **kwargs)
        if self._should_reconstruct_placeholders(**inputs):
            self._construct_placeholders(**inputs)
        elif self.refresh_in_place():
            self._refresh_topology(**inputs)
        with torch.no_grad():
            data = self._update_placeholders(**inputs)
            input_vector = self.construct_input_vector(data, **inputs)
        return data, input_vector

    def _should_reconstruct_placeholders(self, batch_size, **ignored) -> bool:
        refresh = self.refresh_in_place()
        if self.rebuild_every_call and not refresh:
            self._placeholders.clear()
            return True
        cached = self._placeholders.get(batch_size)
        if cached is not None and bool(cached.refreshed_edge_types) == refresh:
            self._example_data = cached
            return False
        if cached is not None:  # built for the other rebuild mode (exact <-> fixed capacity)
            del self._placeholders[batch_size]
        if not self.cache_all_sizes:
            self._placeholders.clear()  # `len(self.example_data) != batch_size` -> rebuild, the old one is dropped
        return True

    def invalidate(self) -> None:
        """Drop every cached topology: the next `build_data` rebuilds it from the batch it is given."""
        self._placeholders.clear()
        self._example_data = None

    # ---- obs splitting (rigid_tasks_data.py:93-150) ---------------------------------------------------
    def _preprocess_input(self, scalars, position_vectors, velocity_vectors, norm_position_vectors,
                          norm_velocity_vectors, infos=None, train: bool = True, **ignored) -> Dict:
        B = scalars.shape[0]
        out = {"batch_size": B, "device": scalars.device, "train": train}

        def split(t, group, as_vec):
            parts = torch.split(t, self.observation_dim[group], dim=1)
            names = self.observation_names[group]
            return {str.__str__(n): (p.reshape(B, -1, 3) if as_vec else p) for n, p in zip(names, parts)}

        out["scalars"] = split(scalars, "scalars", False)
        out["position_vectors"] = split(position_vectors, "position_vectors", True)
        out["velocity_vectors"] = split(velocity_vectors, "velocity_vectors", True)
        out["norm_position_vectors"] = split(norm_position_vectors, "position_vectors", True)
        out["norm_velocity_vectors"] = split(norm_velocity_vectors, "velocity_vectors", True)
        out["infos"] = split(infos, "infos", False) if (infos is not None and self.HAS_INFOS) else {}
        return out

    # ---- topology (K1 kernels) ----------------------------------------------------------------------
    def _num_valid(self, infos, batch_size, device) -> Optional[torch.Tensor]:
        return None

    def _construct_placeholders(self, position_vectors, infos, batch_size, device, **ignored):
        if device.type != "cuda":
            raise RuntimeError("geometry_rl_b200 builds graph topology with CUDA kernels; observations must be on "
                               "a CUDA device (there is no CPU fallback)")
        B = batch_size
        npg = {t: position_vectors[t].shape[1] for t in self.ALL_NODE_TYPES}
        kept = self.node_type_list
        g = GraphBatch(B, {t: npg[t] for t in kept}, device)
        num_valid = self._num_valid(infos, B, device)
        e_int, e_agent, e_task = self.EDGE_TYPES
        P, A = npg[self.PARTICLE_TYPE], npg[self.ACTUATOR_TYPE]
        pts = position_vectors[self.PARTICLE_TYPE]
        refresh = self.refresh_in_place()
        for et in self.EDGE_TYPES:  # insertion order INTERNAL, AGENT, TASK (rigid_tasks_data.py:285-319)
            src, _, dst = et
            if src not in kept or dst not in kept or not self.build_edges:
                continue
            # rewritten in place: what depends on the positions (INTERNAL) or on num_valid (TASK of the rigid tasks)
            refreshed = refresh and (et == e_int or (et == e_task and num_valid is not None))
            if et == e_int and refreshed and self.internal_edges == "knn":
                g.add_edge_set(et, ops.knn_edge_set(pts, num_valid, self.knn_k), refreshed=True)
                continue
            if et == e_int:
                if self.INTERNAL_MODE == "knn" and self.internal_edges == "radius":
                    coo, ptr = self._radius_edges(pts, num_valid, refreshed)
                elif self.INTERNAL_MODE == "knn":
                    coo, ptr = ops.knn_graph(pts, num_valid, self.knn_k)
                else:
                    coo, ptr = ops.dense_edges(0, B, P, P, device)
            elif et == e_agent:
                if A > 1:
                    coo, ptr = ops.dense_edges(0, B, A, A, device)
                else:
                    coo = torch.empty(2, 0, dtype=torch.int64, device=device)
                    ptr = torch.zeros(B + 1, dtype=torch.int64, device=device)
            else:
                coo, ptr = ops.dense_edges(1, B, P, A, device, num_valid=num_valid, capacity=refreshed)
            g.add_edge_type(et, coo, ptr, refreshed=refreshed, exact=not refreshed)
        for t in kept:  # HeteroNodeCategorical: one-hot over the PRE-subgraph type list (transforms.py:43-76)
            oh = torch.zeros(B * npg[t], len(self.ALL_NODE_TYPES), device=device)
            oh[:, list(self.ALL_NODE_TYPES).index(t)] = 1
            g[t].properties = oh
        g.output_mask_key = self._output_mask_key
        g.output_mask = self.output_mask(g, self._output_mask_key)
        self._example_data = g
        self._placeholders[B] = g

    def _radius_edges(self, pts, num_valid, capacity: bool):
        B, P, _ = pts.shape
        return ops.radius_graph(pts, num_valid, self.radius, self.max_num_neighbors,
                                capacity=B * P * self.max_num_neighbors if capacity else None)

    def _refresh_topology(self, position_vectors, infos, batch_size, device, **ignored):
        """Rewrite the refreshed edge types of the cached placeholder from this batch, in place, on the device.

        An edge type with no edge in the whole batch still runs its convolution here (its set has a fixed capacity, so
        emptiness is not visible on the host): every destination row gets the update of an empty neighbourhood, as an
        isolated node does in any batch.  Exact topology (build-once, eager rebuild) skips such an edge type instead,
        as the reference does (hetero_fiber_conv.py:48-49)."""
        g = self._example_data
        num_valid = self._num_valid(infos, batch_size, device)
        e_int = self.EDGE_TYPES[0]
        pts = position_vectors[self.PARTICLE_TYPE]
        for et in g.refreshed_edge_types:
            if et == e_int and self.internal_edges == "knn":
                ops.refresh_knn_edge_set(g.edge_sets[et], pts, num_valid, self.knn_k)
                continue
            if et == e_int:
                coo, ptr = self._radius_edges(pts, num_valid, True)
            else:
                coo, ptr = ops.dense_edges(1, batch_size, pts.shape[1], position_vectors[self.ACTUATOR_TYPE].shape[1],
                                           device, num_valid=num_valid, capacity=True)
            ops.refresh_edge_set(g.edge_sets[et], coo, ptr)
        g.refresh_homogeneous()

    def _update_placeholders(self, position_vectors, norm_position_vectors, device, **ignored) -> GraphBatch:
        data = self._example_data.shallow_copy()
        for t in self.node_type_list:
            data[t].pos = position_vectors[t].reshape(-1, 3)
            data[t].norm_pos = norm_position_vectors[t].reshape(-1, 3)
        return data

    # ---- per-node features ---------------------------------------------------------------------------
    def _vectors(self, data, node_type, norm_position_vectors, norm_velocity_vectors, train) -> torch.Tensor:
        raise NotImplementedError

    def construct_input_vector(self, data: GraphBatch, norm_position_vectors, norm_velocity_vectors, train=True,
                               **ignored):
        scalar_dict, vector_dict, full = {}, {}, {}
        for t in self.node_type_list:
            vectors = self._vectors(data, t, norm_position_vectors, norm_velocity_vectors, train)
            scalar_dict[t] = data[t].properties
            vector_dict[t] = vectors
            if self.concat_input_vector:
                full[t] = torch.cat([data[t].properties, vectors], dim=1)
        return full if self.concat_input_vector else (scalar_dict, vector_dict)

    def _noisy(self, x: torch.Tensor, train: bool) -> torch.Tensor:
        if train and self.training_noise:
            return x + noise_like(x, self.training_noise_std)
        return x
