"""Rigid-body tasks (insertion / pushing / sliding): drop-in for
geometry_rl/modules/pyg_data/rigid_tasks_data.py (same class, enum and constructor names)."""
import enum
from typing import Tuple

import torch

from .base_data import BaseData


class NodeType(str, enum.Enum):
    PARTICLES = "object_geometry"
    ACTUATOR = "grippers"
    TARGET = "target_geometry"


class EdgeLevel(str, enum.Enum):
    INTERNAL = "internal"
    TASK = "task"
    AGENT = "agent"


class EdgeType(Tuple[str, str, str], enum.Enum):
    PARTICLES_INTERNAL_PARTICLES = (NodeType.PARTICLES, EdgeLevel.INTERNAL, NodeType.PARTICLES)
    ACTUATOR_AGENT_ACTUATOR = (NodeType.ACTUATOR, EdgeLevel.AGENT, NodeType.ACTUATOR)
    PARTICLES_TASK_ACTUATOR = (NodeType.PARTICLES, EdgeLevel.TASK, NodeType.ACTUATOR)


class RigidTasksData(BaseData):
    TASK = "rigid"
    ALL_NODE_TYPES = ("object_geometry", "grippers", "target_geometry")
    PARTICLE_TYPE = "object_geometry"
    INTERNAL_MODE = "knn"
    EDGE_TYPES = (("object_geometry", "internal", "object_geometry"), ("grippers", "agent", "grippers"),
                  ("object_geometry", "task", "grippers"))
    HAS_INFOS = True
    HAS_NUM_VALID = True

    def _kept_node_types(self):
        # rigid_tasks_data.py:91: every node type except TARGET
        return [t for t in self.ALL_NODE_TYPES if t != "target_geometry"]

    def _num_valid(self, infos, batch_size, device):
        # rigid_tasks_data.py:272: infos["object_num_points"].long()
        return infos["object_num_points"].reshape(batch_size).to(torch.int32).contiguous()

    def _vectors(self, data, t, npv, nvv, train):
        # rigid_tasks_data.py:170-225
        pos = self._noisy(data[t].norm_pos, train)
        if t == self.PARTICLE_TYPE:
            target = npv["target_geometry"].reshape(-1, 3)
            corr = self._noisy(pos - target if self.dist_as_pos else target, train)
        else:
            corr = torch.zeros_like(pos)
        if t in nvv:
            if t == self.PARTICLE_TYPE:
                n = npv[t].shape[1]
                vel = nvv[t].repeat_interleave(n, dim=1).reshape(-1, 3)
                ang = (nvv[f"{t}_angular"].repeat_interleave(n, dim=1).reshape(-1, 3) if self.angular_velocity
                       else torch.zeros_like(vel))
            else:
                vel = nvv[t].reshape(-1, 3)
                ang = nvv[f"{t}_angular"].reshape(-1, 3) if self.angular_velocity else torch.zeros_like(vel)
            vel, ang = self._noisy(vel, train), self._noisy(ang, train)
        else:
            vel, ang = torch.zeros_like(pos), torch.zeros_like(pos)
        return torch.cat([pos, corr, vel, ang], dim=1)
