"""CPU: the fp64 reference of the 16-bit convolution layer (tests/conv16_reference.py) and its per-row metric.

1. `layer_reference` in float64 agrees with `oracle.models.fiber_bundle_conv + convnext_update` evaluated the way the
   models call them (fibre kernel from the fibre basis MLP, fp32), outputs and gradients, on homogeneous, bipartite and
   sub-layer cases;
2. `row_rel` flags a dropped edge that the global max-norm ratio misses;
3. the longest relative edge vector over the policy graphs of the four message-passing configs, the range the
   dynamic-range test of the kernels scales from."""
import pytest
import torch

from oracle import models as om
from tests import conv16_reference as R
from tests.conv16_reference import LONGEST_EDGE, random_params

MP_CONFIGS = ["rigid_insertion_multi_hepi_trpl_cfg", "rigid_pushing_multi_empn_trpl_cfg", "cloth_hanging_multi_hepi_trpl_cfg",
              "rope_shaping_hepi_trpl_cfg"]


def _oracle_fp32(x_src, x_dst, pos_src, pos_dst, p, fb, fkw, ori, dim, ei, out_ids, g_out):
    """The oracle's layer as hepi_forward calls it, in fp32: fk from the fibre basis, erf GELU; out_ids by slicing."""
    sd = {"basis_fn.1.weight": p["bw1"], "basis_fn.1.bias": p["bb1"], "basis_fn.3.weight": p["bw2"],
          "basis_fn.3.bias": p["bb2"], "c.kernel.weight": p["wk"], "c.fiber_kernel.weight": fkw, "c.bias": p["bias"],
          "c.m.0.weight": p["ln_g"], "c.m.0.bias": p["ln_b"], "c.m.1.weight": p["w1"], "c.m.1.bias": p["b1"],
          "c.m.3.weight": p["w2"], "c.m.3.bias": p["b2"]}
    sp, _ = om.invariants(ori[:, :dim], pos_src[ei[0]][:, :dim], pos_dst[ei[1]][:, :dim])
    kb = om.basis_mlp(sp, sd, "basis_fn")
    xd = x_src if x_dst is None else x_dst
    x2 = om.fiber_bundle_conv(x_src, xd, ei, kb, fb, sd, "c")
    out = om.convnext_update(xd, x2, sd, "c.m.0", "c.m.1", "c.m.3")
    if out_ids is not None:
        out = out[out_ids]
    leaves = [x_src] + ([x_dst] if x_dst is not None else []) + [p[k] for k in R.PARAM_NAMES if k != "fk"] + [fkw]
    return out, torch.autograd.grad(out, leaves, g_out)


@pytest.mark.parametrize("kind", ["homogeneous", "bipartite", "sub"])
@pytest.mark.parametrize("dim", [2, 3])
def test_fp64_reference_matches_oracle_fp32(kind, dim):
    """fp64 vs fp32 of the same operator, so the difference is fp32 rounding alone: within 2e-5 of each tensor's max
    magnitude (measured worst case 1.3e-6), outputs and every gradient, the fibre kernel's through the chain rule."""
    gen = torch.Generator().manual_seed(11 + dim)
    n_src, n_dst, E = 13, (13 if kind != "bipartite" else 5), 40
    p = {k: v.requires_grad_(True) for k, v in random_params(gen).items()}
    x_src = torch.randn(n_src, 16, 64, generator=gen).requires_grad_(True)
    x_dst = torch.randn(n_dst, 16, 64, generator=gen).requires_grad_(True) if kind == "bipartite" else None
    pos_src = torch.randn(n_src, 3, generator=gen) * 0.7
    pos_dst = pos_src if x_dst is None else torch.randn(n_dst, 3, generator=gen) * 0.7
    ei = torch.stack([torch.randint(0, n_src, (E,), generator=gen), torch.randint(0, n_dst, (E,), generator=gen)])
    out_ids = torch.tensor([0, 4, 9]) if kind == "sub" else None
    ori = om.ori_grid(dim, 16)
    ori3 = torch.cat([ori, torch.zeros(16, 3 - dim)], 1)
    fb = torch.randn(16, 16, 3, generator=gen)  # fibre basis (invariant i3 features) -> fk = F.linear(fb, W)
    fkw = (torch.randn(64, 3, generator=gen) * 0.3).requires_grad_(True)
    n_out = n_dst if out_ids is None else 3
    g_out = torch.randn(n_out, 16, 64, generator=gen)
    out32, g32 = _oracle_fp32(x_src, x_dst, pos_src, pos_dst, p, fb, fkw, ori, dim, ei, out_ids, g_out)

    D = torch.float64
    fk = torch.nn.functional.linear(fb.to(D), fkw.detach().to(D))
    p64 = {k: v.detach().to(D) for k, v in p.items()}
    p64["fk"] = fk
    ref = R.layer_reference(x_src.detach().to(D), None if x_dst is None else x_dst.detach().to(D), pos_src.to(D),
                            pos_dst.to(D), p64, ori3.to(D), dim, ei, out_ids=out_ids, grad_out=g_out.to(D))
    names = ["x_src"] + (["x_dst"] if x_dst is not None else []) + [k for k in R.PARAM_NAMES if k != "fk"]
    got = dict(zip(names, g32[:-1]))
    bad = []
    if R.global_rel(out32, ref["out"]) > 2e-5:
        bad.append(f"out {R.global_rel(out32, ref['out']):.2e}")
    for k in names:
        e = R.global_rel(got[k], ref["grad"][k])
        if e > 2e-5:
            bad.append(f"grad {k} {e:.2e}")
    # d/dW of fk = F.linear(fb, W): the reference's grad of fk contracted with fb
    g_fkw = torch.einsum("opc,opf->cf", ref["grad"]["fk"], fb.to(D))
    if R.global_rel(g32[-1], g_fkw) > 2e-5:
        bad.append(f"grad fiber_kernel {R.global_rel(g32[-1], g_fkw):.2e}")
    assert not bad, "\n".join(bad)


def test_row_metric_flags_a_dropped_edge_the_global_metric_misses():
    """A hub destination with 400 coherent in-edges (one source position) and a destination of degree 2: dropping one
    edge of the small node moves x1 by 0.23% of its global max, so the global 1e-2 bound passes; its own row moves by
    about half, which row_rel reports as 0.085 with the default floor (1% of the global max, 11x the row's max here),
    more than 5x that bound."""
    D = torch.float64
    gen = torch.Generator().manual_seed(3)
    p = random_params(gen, D)
    n_src = 402
    x_src = torch.randn(n_src, 16, 64, generator=gen, dtype=D)
    x_src[:400] = x_src[0]  # coherent messages: the hub's row grows linearly with its degree
    pos_src = torch.randn(n_src, 3, generator=gen, dtype=D) * 0.5
    pos_src[:400] = pos_src[0]
    pos_dst = torch.randn(2, 3, generator=gen, dtype=D) * 0.5
    ei = torch.stack([torch.arange(402), torch.tensor([0] * 400 + [1, 1])])
    ori3 = torch.cat([om.ori_grid(3, 16).to(D), torch.zeros(16, 0, dtype=D)], 1)
    kw = dict(x_src=x_src, pos_src=pos_src, pos_dst=pos_dst, params=p, ori3=ori3, dim=3, n_dst=2)
    ref = R.edge_reference(edge_index=ei, **kw)["x1"]
    dropped = R.edge_reference(edge_index=R.perturbation(ei, "drop", n_src), **kw)["x1"]
    assert R.global_rel(dropped, ref) < 1e-2
    assert R.row_rel(dropped, ref) > 5e-2
    assert R.row_rel(dropped, ref, floor=0.0) > 0.3
    # and the edge it dropped is the last in-edge of the degree-2 node
    assert R.perturbation(ei, "drop", n_src).shape[1] == 401 and float((dropped[0] - ref[0]).abs().max()) == 0.0


def test_perturbation_picks_the_last_edge_at_a_tile_boundary():
    # degrees 2, 4, 2, 8, 1 in dst-sorted order: the nodes end at entries 1, 5, 7, 15, 16; of the two nodes of degree 2
    # (degree 1 has no second edge) the one ending the first tile of 8 (node 2, entry 7) loses its last edge
    dst = torch.tensor([0] * 2 + [1] * 4 + [2] * 2 + [3] * 8 + [4])
    src = torch.arange(17)
    ei = torch.stack([src, dst])
    d = R.perturbation(ei, "drop", 17)
    assert d.shape[1] == 16 and 7 not in d[0].tolist()
    s = R.perturbation(ei, "swap", 17)
    assert int((s != ei).sum()) == 1 and s[1].equal(ei[1]) and int(s[0, 7]) != 7


def test_longest_edge_of_the_synthetic_observations():
    """The longest relative edge vector of the four message-passing configs' policy graphs (kNN internal edges, TASK
    and AGENT edges, as the data builders make them): measured 1.8141, recorded as conv16_reference.LONGEST_EDGE."""
    from oracle import graph as og
    from geometry_rl_b200.synthetic import CONFIGS, obs_keys, observation_layout, synthetic_obs
    longest = 0.0
    for name in MP_CONFIGS:
        cfg = CONFIGS[name]
        gen = torch.Generator().manual_seed(0)
        B = 64
        obs = synthetic_obs(cfg, B, gen, env_ids=torch.arange(B) * max(1, cfg.num_envs // B) % cfg.num_envs)
        dims, names = observation_layout(cfg)
        parts = og.split_obs({k: obs[k] for k in obs_keys(cfg)}, dims, names)
        num_points = parts["infos"]["object_num_points"].long().reshape(-1) if cfg.task == "rigid" else None
        g = og.build_topology(og.TASKS[cfg.task], parts["position_vectors"], full_graph_obs=False,
                              output_mask_key="grippers", num_points=num_points)
        og.update_positions(g, parts["position_vectors"], parts["norm_position_vectors"])
        for (s, _, d), ei in g.edge_index_dict.items():
            if ei.numel():
                rel = g.pos[s][ei[0]][:, :cfg.ponita_dim] - g.pos[d][ei[1]][:, :cfg.ponita_dim]
                longest = max(longest, float(rel.norm(dim=1).max()))
    assert 0.0 < longest <= LONGEST_EDGE, f"longest edge {longest:.4f}: update conv16_reference.LONGEST_EDGE"
    assert longest > 0.9 * LONGEST_EDGE, f"longest edge {longest:.4f}: update conv16_reference.LONGEST_EDGE"
