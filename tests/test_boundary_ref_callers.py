"""CPU, optional (needs a thobotics/geometry_rl checkout named by $GRL_REFERENCE): the reference's OWN wrapper classes
accept the repo's bodies and data builders — the duck-typed drop-in INTEGRATION.md section 1 describes.

The unmodified `GNNGaussianPolicyDiag` / `GNNVFNet` are imported from that checkout through oracle/ref_shims and
constructed around the repo's `HEPi` / `DeepSets` / `RigidTasksData` objects.  There is no GPU here, so the bodies cannot
execute; what is checked is everything the wrapper itself touches: constructor contract (`gnn.device`), parameter
registration (state_dict keys equal the ones the all-reference wrapper saved in the fixture), and the call protocol
`hyper_data.build_data(*obs, train=) -> gnn.one_step(graph, input_vector)` with the argument order and keywords the
reference uses (abstract_gnn_gaussian_policy.py:95-109, value/gnn_vf_net.py:88-102).  The numeric half of the same
boundary runs on the GPU against fixtures from the all-reference stack: tests/test_gpu_boundary.py."""
import os
import sys

import pytest
import torch

REF = os.environ.get("GRL_REFERENCE", "")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "geometry_rl")),
                                reason="set GRL_REFERENCE to a thobotics/geometry_rl checkout to run the reference's own wrappers")


@pytest.fixture(scope="module")
def ref_paths():
    added = [os.path.join(ROOT, "oracle", "ref_shims"), REF]
    for p in added:
        sys.path.insert(0, p)
    yield
    for p in added:
        sys.path.remove(p)


def _repo_objects(cfg, policy):
    from geometry_rl_b200 import learner
    body = learner.make_policy_body(cfg, "cpu") if policy else None
    return body, learner.make_data(cfg, policy=policy)


def test_reference_policy_wrapper_drives_the_repo_body(ref_paths):
    from geometry_rl.algorithms.trust_region_projections.models.policy.gnn_gaussian_policy_diag import (
        GNNGaussianPolicyDiag as RefPolicy)
    from geometry_rl_b200.synthetic import CONFIGS
    from tests.helpers import load_golden
    cfg = CONFIGS["rigid_insertion_multi_hepi_trpl_cfg"]
    body, data = _repo_objects(cfg, policy=True)
    pol = RefPolicy(gnn=body, hyper_data=data, action_dim=cfg.total_action_dim, num_actuators=cfg.num_actuators,
                    init="orthogonal", hidden_sizes=(64, 64), contextual_std=True, init_std=1.0, minimal_std=1e-5,
                    share_action_dim=True, post_fc=cfg.post_fc)
    fixture = load_golden("policy_wrapper_rigid_insertion")
    assert set(pol.state_dict().keys()) == set(fixture["state_dict"].keys())
    for k, v in pol.state_dict().items():
        assert tuple(v.shape) == tuple(fixture["state_dict"][k].shape), k
    pol.load_state_dict(fixture["state_dict"], strict=True)  # a reference checkpoint loads into reference-wrapper + repo body

    calls = {}
    B, A = 4, cfg.num_actuators

    def build_data(*args, train=True):
        calls["build"] = (len(args), train)
        return "graph", "features"

    def one_step(graph, input_vector):
        calls["step"] = (graph, input_vector)
        return torch.zeros(B * A * cfg.output_dim_vec, 3), torch.zeros(B * A, 64)

    data.build_data, body.one_step = build_data, one_step
    obs = [torch.zeros(B, 3)] * 6
    loc, cov = pol(*obs, train=False)
    assert calls["build"] == (6, False) and calls["step"] == ("graph", "features")
    assert loc.shape == (B, cfg.total_action_dim) and cov.shape == (B, cfg.total_action_dim, cfg.total_action_dim)


def test_reference_value_wrapper_drives_the_repo_critic(ref_paths):
    from geometry_rl.algorithms.trust_region_projections.models.value.gnn_vf_net import GNNVFNet as RefVF
    from geometry_rl_b200.modules.pyg_models.deepsets import DeepSets
    from geometry_rl_b200.synthetic import CONFIGS
    from tests.helpers import load_golden
    cfg = CONFIGS["rigid_insertion_multi_hepi_trpl_cfg"]
    _, data = _repo_objects(cfg, policy=False)
    gnn = DeepSets(input_dim_node=3 + 12, output_dim=64, hidden_dim=64, norm=["layer_norm", "layer_norm"])
    vf = RefVF(gnn=gnn, hyper_data=data, init="orthogonal", hidden_sizes=(64, 64))
    fixture = load_golden("value_wrapper_rigid")
    assert set(vf.state_dict().keys()) == set(fixture["state_dict"].keys())
    vf.load_state_dict(fixture["state_dict"], strict=True)
    seen = []
    data.build_data = lambda *a, train=True: (seen.append((len(a), a[0].shape, train)) or ("g", "f"))
    gnn.one_step = lambda g, f: torch.zeros(5, 64)
    v = vf(*[torch.zeros(5, 2, 7)] * 6)  # 3-D observations: the reference loops over time and calls the body per step
    assert v.shape == (5, 2, 1) and seen == [(6, torch.Size([5, 7]), True)] * 2
