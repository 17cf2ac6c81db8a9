"""GPU: the four kernels of the benched 16-bit convolution layer (FusedFiberConvFn) against the fp64 reference of
tests/conv16_reference.py, with a per-row metric, at tile, segment and capacity edges.

a. grl_fbconv_edge_fused_fwd / _bwd alone, through the C ABI: x1, grad_x_src and the gradients of wk and of the basis
   MLP; hub nodes, entry counts = 0, 1, 7 mod 8, a one-row tensor map, more CTAs than key nodes with edges, both dims,
   bipartite sets and the data builders' topologies; exact zeros / init rows, repeatability, capacity tails never read,
   every valid partial count;
b. grl_fbconv_node_fwd_tc / grl_fbconv_node_bwd_tc alone, through the C ABI, fed a random x1: out, x2, grad_x1 and the
   eight node gradients around the launch grid's tile counts, every partial count, the fp16 gradient scale and
   accumulate_out;
c. the whole layer, ops.fiber_conv with a BasisSpec: homogeneous, bipartite, sub layer, capacity radius graph with an
   all-empty graph, and the benchmark's rope topology at minibatch 2048;
d. loss-scale covariance of the fused path (exact for powers of two);
e. dynamic range: long edges and small weights.

Every output and partial buffer is filled with NaN before a launch.  Every case also evaluates the reference on an
edge list with one edge dropped and one with one source swapped (conv16_reference.perturbed) and asserts that the
per-row metric puts that at 5x or more of the tolerance, so the tolerance is shown to catch a lost or misrouted edge.
None of these tests uses the materialised-basis kernels or the strict fp32 path.

Tolerances are per-row (conv16_reference.row_rel, floor 1% of the tensor's max) and were set from the worst case
measured on one B200 with headroom; the global max-norm bound of north_star (1e-2) is asserted as well."""
import ctypes as C

import pytest
import torch

from tests import conv16_reference as R
from tests import gpu_helpers as G
from tests.conv16_reference import LONGEST_EDGE, random_params

pytestmark = pytest.mark.gpu

D = torch.float64
NAN = float("nan")
# Per-row tolerances (row_rel, floor 1e-2) of the node tensors, [N,16,64]; a row is one node at one orientation.  Worst
# cases measured on one B200 (1000 W power limit) over every case of this file:
TOL_X1 = 2e-2         # x1 of the fused edge forward: 9.9e-3 (bipartite)
TOL_GXS = 3e-2        # grad_x_src of the fused edge backward: 1.8e-2 (whole layer, sub)
TOL_OUT = 1.5e-2      # layer output minus the residual: 7.1e-3 (whole layer, homogeneous)
TOL_GX1 = 1e-2        # grad_x1 of the node backward: 3.6e-3 (n_dst 20011)
TOL_X2 = 1e-5         # x2 = fibre(x1) + bias, fp32 work: 3.7e-7
# Weight gradients are sums over every edge or node, not rows of a node tensor: global max-norm bounds.
GLOBAL = 1e-2         # north_star's bound, max|a-b| / max|b|: worst 5.3e-3 (wk), every node and output tensor below it
GLOBAL_BASIS = 2.5e-2  # basis-MLP gradients (three chained bf16 roundings), as in test_gpu_fused.py: worst 1.1e-2 (bb1)
BASIS = ("bw1", "bb1", "bw2", "bb2")
EDGE_SIDE = ("x_src", "wk") + BASIS  # gradients that leave the fused edge backward


def _ori(dim):
    from geometry_rl_b200.modules.pyg_models.ponita.ponita import make_ori_grid, pad_ori3
    return pad_ori3(make_ori_grid(dim, 16, False).cuda())


def _params(seed, wk_scale=0.12, bw2_scale=0.15):
    return {k: v.cuda() for k, v in random_params(torch.Generator().manual_seed(seed), torch.float32, wk_scale,
                                                   bw2_scale).items()}


class Topo:
    """A key-sorted entry list in both orders, as the fused kernels take it: dst-sorted (edge order, ties in COO order)
    and src-sorted (ties in edge order), with their CSR row pointers; `ei` is the edge list for the reference."""

    def __init__(self, src, dst, n_src, n_dst):
        src, dst = src.long().cuda(), dst.long().cuda()
        o = torch.sort(dst, stable=True).indices
        self.e_src, self.e_dst = src[o].int().contiguous(), dst[o].int().contiguous()
        o2 = torch.sort(self.e_src.long(), stable=True).indices
        self.s_src, self.s_dst = self.e_src[o2].contiguous(), self.e_dst[o2].contiguous()
        self.rowptr_dst = self._rowptr(self.e_dst, n_dst)
        self.rowptr_src = self._rowptr(self.s_src, n_src)
        self.n_src, self.n_dst, self.n_edges = n_src, n_dst, int(src.numel())
        self.ei = torch.stack([self.e_src.long(), self.e_dst.long()])

    @staticmethod
    def _rowptr(keys, n):
        rp = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
        rp[1:] = torch.cumsum(torch.bincount(keys.long(), minlength=n), 0)
        return rp.int().contiguous()

    @classmethod
    def of_edge_set(cls, es):
        from geometry_rl_b200 import ops
        es = ops.exact_edge_set(es)
        return cls(es.edge_src, es.edge_dst, es.n_src, es.n_dst)


def _edge_fwd(t, pos_src, pos_dst, p, x_src, dim, e_src=None, e_dst=None, n_edges=None):
    from geometry_rl_b200 import _lib as L
    x1 = torch.full((t.n_dst, 16, 64), NAN, device="cuda")
    fd = L.GrlFusedEdgeDesc(n_key=t.n_dst, n_other=t.n_src, n_edges=t.n_edges if n_edges is None else n_edges, dim=dim,
                            n_partials=0, rowptr=L.ptr(t.rowptr_dst), e_src=L.ptr(t.e_src if e_src is None else e_src),
                            e_dst=L.ptr(t.e_dst if e_dst is None else e_dst), pos_src=L.ptr(pos_src),
                            pos_dst=L.ptr(pos_dst), ori=L.ptr(_ori(dim)), w1=L.ptr(p["bw1"]), b1=L.ptr(p["bb1"]),
                            w2=L.ptr(p["bw2"]), b2=L.ptr(p["bb2"]), wk=L.ptr(p["wk"]), x_src=L.ptr(x_src), x1=L.ptr(x1))
    L.call("grl_fbconv_edge_fused_fwd", C.byref(fd))
    return x1


def _edge_bwd(t, pos_src, pos_dst, p, x_src, g_x1, dim, n_p, init=None, s_src=None, s_dst=None, n_edges=None):
    from geometry_rl_b200 import _lib as L
    g_xs = torch.full((t.n_src, 16, 64), NAN, device="cuda")
    part = torch.full((n_p, L.FUSED_EDGE_GRAD_FLOATS), NAN, device="cuda")
    bd = L.GrlFusedEdgeDesc(n_key=t.n_src, n_other=t.n_dst, n_edges=t.n_edges if n_edges is None else n_edges, dim=dim,
                            n_partials=n_p, rowptr=L.ptr(t.rowptr_src), e_src=L.ptr(t.s_src if s_src is None else s_src),
                            e_dst=L.ptr(t.s_dst if s_dst is None else s_dst), pos_src=L.ptr(pos_src),
                            pos_dst=L.ptr(pos_dst), ori=L.ptr(_ori(dim)), w1=L.ptr(p["bw1"]), b1=L.ptr(p["bb1"]),
                            w2=L.ptr(p["bw2"]), b2=L.ptr(p["bb2"]), wk=L.ptr(p["wk"]), x_src=L.ptr(x_src),
                            grad_x1=L.ptr(g_x1), grad_x_src=L.ptr(g_xs), grad_x_src_init=L.ptr(init),
                            grad_partials=L.ptr(part))
    L.call("grl_fbconv_edge_fused_bwd", C.byref(bd))
    return g_xs, part


def _unpack_edge(part):
    ge = part.double().sum(0)
    w1b = ge[4096:5120].view(64, 16)
    return {"wk": ge[:4096].view(64, 64), "bw1": w1b[:, :14], "bb1": w1b[:, 14], "bw2": ge[5120:9216].view(64, 64),
            "bb2": ge[9216:9280]}


def _check(bad, name, got, ref, tol, report):
    """A node tensor: per-row `tol` and the global bound."""
    r, g = R.row_rel(got, ref), R.global_rel(got, ref)
    report.append(f"{name}: row {r:.3e} global {g:.3e}")
    if not (r < tol and g < GLOBAL):
        bad.append(f"{name}: row {r:.3e} (tol {tol:g}) global {g:.3e}")


def _check_weight(bad, name, got, ref, report):
    """A weight gradient: the global bound (GLOBAL_BASIS for the basis MLP)."""
    tol = GLOBAL_BASIS if name.split()[-1] in BASIS else GLOBAL
    g = R.global_rel(got, ref)
    report.append(f"{name}: global {g:.3e}")
    if not g < tol:
        bad.append(f"{name}: global {g:.3e} (tol {tol:g})")


# ---------------------------------------------------------------------------------------------------------------------
# a. fused edge kernels alone
# ---------------------------------------------------------------------------------------------------------------------
def _edge_case(name):
    """(src, dst, n_src, n_dst, dim, pos scale).  Every case keeps some key nodes without edges on both sides."""
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    ri = lambda hi, n: torch.randint(0, hi, (n,), generator=g)  # noqa: E731
    if name == "hub_dst":  # one destination with in-degree 5000: one CTA's range is one node spanning 625 tiles
        src = torch.cat([torch.arange(5000), torch.tensor([0, 1, 2, 3, 4])])
        dst = torch.cat([torch.zeros(5000, dtype=torch.long), torch.tensor([1, 1, 2, 2, 2])])
        return src, dst, 5002, 4, 3
    if name == "hub_src":  # one source with out-degree 5000 (the backward's key side)
        src = torch.cat([torch.zeros(5000, dtype=torch.long), torch.tensor([1, 1, 2])])
        dst = torch.cat([torch.arange(5000), torch.tensor([0, 7, 7])])
        return src, dst, 4, 5002, 3
    if name.startswith("mod8"):  # key ranges of 0, 1, 7, 8, 9, 15, 16, 17 entries, both sides
        degs = torch.tensor([8, 9, 15, 0, 1, 7, 16, 17, 2] * 6)
        dst = torch.repeat_interleave(torch.arange(degs.numel()), degs)
        src = torch.repeat_interleave(torch.arange(degs.numel()), degs.roll(4))[torch.randperm(dst.numel(), generator=g)]
        return src, dst, degs.numel(), degs.numel(), int(name[-1])
    if name == "one_src_row":  # n_other = 1 in the forward: a one-row tensor map over x_src
        dst = torch.cat([torch.arange(3000), torch.arange(10)])
        return torch.zeros(dst.numel(), dtype=torch.long), dst, 1, 3001, 3
    if name == "one_dst_row":  # n_other = 1 in the backward: a one-row tensor map over grad_x1
        return torch.arange(3000), torch.zeros(3000, dtype=torch.long), 3001, 1, 2
    if name == "sparse_keys":  # 2000 key nodes, 5 with edges: more CTAs than nodes that have work
        dst = torch.repeat_interleave(torch.tensor([3, 500, 501, 1200, 1999]), torch.tensor([3, 2, 40, 1, 9]))
        return ri(300, dst.numel()), dst, 300, 2000, 3
    if name == "bipartite":
        return ri(700, 4000), ri(300, 4000), 703, 300, 2
    raise KeyError(name)


def _builder_topology(kind):
    """Edge sets the data builders make: rope kNN and radius internal edges, rigid TASK edges at minibatch 1024."""
    from geometry_rl_b200.synthetic import CONFIGS, observation_layout, synthetic_obs
    name = "rope_shaping_hepi_trpl_cfg" if kind.startswith("rope") else "rigid_insertion_multi_hepi_trpl_cfg"
    cfg = CONFIGS[name]
    B = 64 if kind.startswith("rope") else 1024
    obs = synthetic_obs(cfg, B, torch.Generator().manual_seed(21), env_ids=torch.arange(B) % cfg.num_envs)
    data = G.make_data(cfg, policy=True)
    if kind == "rope_radius":  # rope links sit ~0.010 apart: radius 0.025 gives degree ~4, at most 8 neighbours
        dims, names = observation_layout(cfg)
        data = type(data)(observation_dim=dims, observation_names=names, full_graph_obs=False, dist_as_pos=True,
                          output_mask_key="grippers", concat_input_vector=False, angular_velocity=cfg.angular_velocity,
                          internal_edges="radius", radius=0.025, max_num_neighbors=8)
    graph, _ = data.build_data(*G.obs_args(cfg, obs, policy=True), train=False)
    et = ("links", "internal", "links") if kind.startswith("rope") else ("object_geometry", "task", "grippers")
    es = graph.edge_sets[et]
    return Topo.of_edge_set(es), graph[et[0]].pos.float().contiguous(), graph[et[2]].pos.float().contiguous(), \
        cfg.ponita_dim


EDGE_CASES = ["hub_dst", "hub_src", "mod8_dim2", "mod8_dim3", "one_src_row", "one_dst_row", "sparse_keys", "bipartite",
              "rope_knn", "rope_radius", "rigid_task"]


@pytest.mark.parametrize("name", EDGE_CASES)
def test_fused_edge_kernels_alone_against_fp64(name):
    from geometry_rl_b200 import _lib as L
    if name in ("rope_knn", "rope_radius", "rigid_task"):
        t, pos_src, pos_dst, dim = _builder_topology(name)
    else:
        src, dst, ns, nd, dim = _edge_case(name)
        t = Topo(src, dst, ns, nd)
        gp = torch.Generator().manual_seed(5)
        pos_src = (torch.randn(ns, 3, generator=gp) * 0.6).cuda()
        pos_dst = (torch.randn(nd, 3, generator=gp) * 0.6).cuda()
    g = torch.Generator().manual_seed(17)
    x_src = torch.randn(t.n_src, 16, 64, generator=g).cuda()
    g_x1 = torch.randn(t.n_dst, 16, 64, generator=g).cuda()
    init = torch.randn(t.n_src, 16, 64, generator=g).cuda() if t.n_src % 2 == 0 else None
    p = _params(3)
    n_p = max(1, min(t.n_src, L.sm_count()))

    x1 = _edge_fwd(t, pos_src, pos_dst, p, x_src, dim)
    g_xs, part = _edge_bwd(t, pos_src, pos_dst, p, x_src, g_x1, dim, n_p, init)
    torch.cuda.synchronize()

    ref_kw = dict(x_src=x_src.to(D), pos_src=pos_src.to(D), pos_dst=pos_dst.to(D), params=p, ori3=_ori(dim).to(D),
                  dim=dim, n_dst=t.n_dst, grad_x1=g_x1.to(D))
    ref = R.edge_reference(edge_index=t.ei, **ref_kw)
    ref_gxs = ref["grad"]["x_src"] + (init.to(D) if init is not None else 0)
    got = _unpack_edge(part)
    bad, report = [], []
    _check(bad, "x1", x1, ref["x1"], TOL_X1, report)
    _check(bad, "grad_x_src", g_xs, ref_gxs, TOL_GXS, report)
    for k in ("wk",) + BASIS:
        _check_weight(bad, f"grad {k}", got[k], ref["grad"][k], report)
    print(f"[edge {name}] " + "; ".join(report))
    assert not bad, "\n".join(bad)

    # exact: rows without an edge
    no_in = (t.rowptr_dst[1:] == t.rowptr_dst[:-1])
    no_out = (t.rowptr_src[1:] == t.rowptr_src[:-1])
    assert bool((x1[no_in] == 0).all()), "x1 rows of nodes without an in-edge must be exactly 0"
    want = init[no_out] if init is not None else torch.zeros_like(g_xs[no_out])
    assert torch.equal(g_xs[no_out], want), "grad_x_src rows of sources without an out-edge must equal the init (or 0)"

    # exact: a second launch gives the same bits, outputs and partials
    x1b = _edge_fwd(t, pos_src, pos_dst, p, x_src, dim)
    g_xsb, partb = _edge_bwd(t, pos_src, pos_dst, p, x_src, g_x1, dim, n_p, init)
    assert torch.equal(x1, x1b) and torch.equal(g_xs, g_xsb) and torch.equal(part, partb), "not repeatable"

    # every valid partial count: the same grad_x_src bits; the summed partials differ by fp32 reassociation only.  One
    # CTA accumulating every edge in fp32 (n_partials = 1) moves grad wk by up to 4.9e-4 of its max (rigid TASK edges),
    # about n * 2^-24 for the ~5000 tiles' worth of cancelling terms; held to 2e-3 and, like every count, to the bounds
    for n_pp in sorted({1, min(7, t.n_src), t.n_src}):
        g_xs2, part2 = _edge_bwd(t, pos_src, pos_dst, p, x_src, g_x1, dim, n_pp, init)
        assert torch.equal(g_xs2, g_xs), f"grad_x_src depends on n_partials={n_pp}"
        got2 = _unpack_edge(part2)
        for k, v in got2.items():
            e = R.global_rel(v, got[k])
            assert e < 2e-3, f"n_partials={n_pp}: grad {k} moved by {e:.2e} of its max"
            _check_weight(bad, f"n_partials={n_pp} grad {k}", v, ref["grad"][k], report)
    assert not bad, "\n".join(bad)

    # the tolerance catches one dropped / one misrouted edge (forward x1 or backward grad_x_src, whichever the case's
    # topology lets one edge dominate a row of)
    kinds = ("drop", "swap") if t.n_src >= 2 else ("drop",)
    for kind in kinds:
        pe = R.edge_reference(edge_index=R.perturbation(t.ei, kind, t.n_src), **ref_kw)
        pg = pe["grad"]["x_src"] + (init.to(D) if init is not None else 0)
        r1, r2 = R.row_rel(pe["x1"], ref["x1"]), R.row_rel(pg, ref_gxs)
        assert max(r1 / TOL_X1, r2 / TOL_GXS) >= 5, f"one {kind} edge: x1 {r1:.3e}, grad_x_src {r2:.3e}"


@pytest.mark.parametrize("name", ["hub_dst", "mod8_dim3", "sparse_keys", "rope_radius"])
def test_fused_edge_kernels_never_read_past_the_real_edge_count(name):
    """The same entry list padded to a capacity: n_edges = capacity, the tail of e_src / e_dst filled with valid ids of
    OTHER real nodes.  x1, grad_x_src and every partial slot are bit-identical to the exact-size launch."""
    from geometry_rl_b200 import _lib as L
    if name == "rope_radius":
        t, pos_src, pos_dst, dim = _builder_topology(name)
    else:
        src, dst, ns, nd, dim = _edge_case(name)
        t = Topo(src, dst, ns, nd)
        gp = torch.Generator().manual_seed(5)
        pos_src = (torch.randn(ns, 3, generator=gp) * 0.6).cuda()
        pos_dst = (torch.randn(nd, 3, generator=gp) * 0.6).cuda()
    g = torch.Generator().manual_seed(29)
    x_src = torch.randn(t.n_src, 16, 64, generator=g).cuda()
    g_x1 = torch.randn(t.n_dst, 16, 64, generator=g).cuda()
    p = _params(4)
    cap = t.n_edges + 8 * 37 + 5
    pad = cap - t.n_edges
    tail_src = torch.randint(0, t.n_src, (pad,), generator=g).int().cuda()
    tail_dst = torch.randint(0, t.n_dst, (pad,), generator=g).int().cuda()
    pad_e = lambda a, tail: torch.cat([a, tail]).contiguous()  # noqa: E731
    for n_p in sorted({1, min(7, t.n_src), max(1, min(t.n_src, L.sm_count()))}):
        x1 = _edge_fwd(t, pos_src, pos_dst, p, x_src, dim)
        x1c = _edge_fwd(t, pos_src, pos_dst, p, x_src, dim, pad_e(t.e_src, tail_src), pad_e(t.e_dst, tail_dst), cap)
        gx, part = _edge_bwd(t, pos_src, pos_dst, p, x_src, g_x1, dim, n_p)
        gxc, partc = _edge_bwd(t, pos_src, pos_dst, p, x_src, g_x1, dim, n_p, s_src=pad_e(t.s_src, tail_src),
                               s_dst=pad_e(t.s_dst, tail_dst), n_edges=cap)
        assert torch.equal(x1, x1c), "the forward read entries past rowptr[n_key]"
        assert torch.equal(gx, gxc) and torch.equal(part, partc), f"the backward read entries past rowptr[n_key] (n_p={n_p})"


# ---------------------------------------------------------------------------------------------------------------------
# b. tensor-core node kernels alone
# ---------------------------------------------------------------------------------------------------------------------
def _node_launch(n_dst, x1, x_dst, p, g_out, n_pn, amax_mode="absmax", accumulate=None, with_x2=True):
    from geometry_rl_b200 import _lib as L
    out = torch.full((n_dst, 16, 64), NAN, device="cuda") if accumulate is None else accumulate.clone()
    x2 = torch.full((n_dst, 16, 64), NAN, device="cuda") if with_x2 else None
    d = L.GrlConvDesc(n_src=n_dst, n_dst=n_dst, n_edges=0, x_src=L.ptr(x1), x_dst=L.ptr(x_dst), fiber_kernel=L.ptr(p["fk"]),
                      wk=L.ptr(p["wk"]), bias=L.ptr(p["bias"]), ln_g=L.ptr(p["ln_g"]), ln_b=L.ptr(p["ln_b"]),
                      w1=L.ptr(p["w1"]), b1=L.ptr(p["b1"]), w2=L.ptr(p["w2"]), b2=L.ptr(p["b2"]), x1=L.ptr(x1),
                      out=L.ptr(out), accumulate_out=int(accumulate is not None), x2=L.ptr(x2),
                      wk_t=L.ptr(p["wk"]), w1_t=L.ptr(p["w1"]), w2_t=L.ptr(p["w1"]), w2_c=L.ptr(p["w1"]))
    L.call("grl_fbconv_node_fwd_tc", C.byref(d))
    if g_out is None:
        return out, x2, None, None
    amax = None
    if amax_mode == "absmax":
        amax = torch.empty(1, dtype=torch.int32, device="cuda")
        L.call("grl_absmax", L.ptr(g_out), g_out.numel(), L.ptr(amax))
    g_x1 = torch.full_like(x1, NAN)
    g_x2 = torch.full_like(x1, NAN)
    part = torch.full((n_pn, L.NODE_GRAD_FLOATS), NAN, device="cuda")
    d.grad_out, d.grad_x1, d.grad_x2, d.grad_amax = L.ptr(g_out), L.ptr(g_x1), L.ptr(g_x2), L.ptr(amax)
    d.node_grad_partials, d.n_partials_node = L.ptr(part), n_pn
    L.call("grl_fbconv_node_bwd_tc", C.byref(d))
    return out, x2, g_x1, part


NODE_SLICES = [("w1", 256 * 64, (256, 64)), ("b1", 256, (256,)), ("w2", 64 * 256, (64, 256)), ("b2", 64, (64,)),
               ("ln_g", 64, (64,)), ("ln_b", 64, (64,)), ("bias", 64, (64,)), ("fk", 16 * 16 * 64, (16, 16, 64))]


def _unpack_node(part):
    g, o, res = part.double().sum(0), 0, {}
    for k, n, shape in NODE_SLICES:
        res[k] = g[o:o + n].view(shape)
        o += n
    return res


def _node_reference(x1, x_dst, p, g_out):
    """The reference's node half: the layer with one identity message per node (kernel.weight = I, a basis of ones),
    so that its x1 is the given x1 and its grad of x_src is grad_x1."""
    n = x1.shape[0]
    pr = dict(p, wk=torch.eye(64, dtype=D, device="cuda"))
    ei = torch.arange(n, device="cuda").expand(2, -1)
    return R.layer_reference(x1.to(D), x_dst.to(D), x1.to(D)[:, 0, :3], x1.to(D)[:, 0, :3], pr, _ori(3).to(D), 3, ei,
                             grad_out=None if g_out is None else g_out.to(D),
                             kernel_basis=torch.ones(n, 16, 64, dtype=D, device="cuda"))


def _assert_node_perturbation_caught(x1, x_dst, p, ref, g_out=None):
    """The node kernels see no edges, so the stand-in for a lost message is one node losing half of its input: half of
    one orientation row of x1 (what dropping one of two in-edges does to it) must move `out` by >= 5x TOL_OUT, and half
    of the node's upstream gradient must move its grad_x1 row by >= 5x TOL_GX1."""
    k = x1.shape[0] // 2
    pd = {n: v.to(D) for n, v in p.items()}
    x1p = x1.clone()
    x1p[k, 5] *= 0.5
    r = R.row_rel(_node_reference(x1p, x_dst, pd, None)["out"] - x_dst.to(D), ref["out"] - x_dst.to(D))
    assert r >= 5 * TOL_OUT, f"half a message moves out by {r:.3e} only"
    if g_out is not None:
        gp = g_out.clone()
        gp[k] *= 0.5
        r = R.row_rel(_node_reference(x1, x_dst, pd, gp)["grad"]["x_src"], ref["grad"]["x_src"])
        assert r >= 5 * TOL_GX1, f"half a node's upstream gradient moves grad_x1 by {r:.3e} only"


def _node_inputs(n_dst, seed=41):
    g = torch.Generator().manual_seed(seed)
    x1 = (torch.randn(n_dst, 16, 64, generator=g) * 2).cuda()
    x_dst = torch.randn(n_dst, 16, 64, generator=g).cuda()
    g_out = torch.randn(n_dst, 16, 64, generator=g).cuda()
    return x1, x_dst, g_out


def _grid():
    from geometry_rl_b200 import _lib as L
    return L.sm_count()


def _node_sizes():
    G2 = 8 * 2 * _grid()
    return [1, 7, 8, 9, 16, 17, G2 - 8, G2, G2 + 8, 20011]


@pytest.mark.parametrize("idx", range(10), ids=["1", "7", "8", "9", "16", "17", "16G-8", "16G", "16G+8", "20011"])
def test_node_kernels_alone_against_fp64(idx):
    n_dst = _node_sizes()[idx]
    x1, x_dst, g_out = _node_inputs(n_dst)
    p = _params(8)
    n_tiles = (n_dst + 7) // 8
    ref = _node_reference(x1, x_dst, {k: v.to(D) for k, v in p.items()}, g_out)
    report, bad = [], []
    first = None
    for n_pn in sorted({1, 5, n_tiles, n_tiles + 3}):
        out, x2, g_x1, part = _node_launch(n_dst, x1, x_dst, p, g_out, n_pn)
        again = _node_launch(n_dst, x1, x_dst, p, g_out, n_pn)
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip((out, x2, g_x1, part), again)), "two identical launches differ"
        if first is None:
            first = (out, x2, g_x1)
            _check(bad, "out - x_dst", out - x_dst, ref["out"] - x_dst.to(D), TOL_OUT, report)
            _check(bad, "x2", x2, ref["x2"], TOL_X2, report)
            _check(bad, "grad_x1", g_x1, ref["grad"]["x_src"], TOL_GX1, report)
        else:
            assert torch.equal(out, first[0]) and torch.equal(x2, first[1])
            assert torch.equal(g_x1, first[2]), f"grad_x1 depends on n_partials_node={n_pn}"
        got = _unpack_node(part)
        for k, _, _ in NODE_SLICES:
            _check_weight(bad, f"n_p={n_pn} grad {k}", got[k], ref["grad"][k], report)
        # slots of CTAs that get no tile hold exact zeros: no 8-node MLP tile past n_tiles, no 4-node fibre tile past
        # (n_dst + 3) // 4
        mlp_floats = sum(n for k, n, _ in NODE_SLICES[:6])
        assert bool((part[n_tiles:, :mlp_floats] == 0).all()), "an idle CTA's MLP partial slot is not zero"
        assert bool((part[(n_dst + 3) // 4:] == 0).all()), "an idle CTA's partial slot is not zero"
    print(f"[node {n_dst}] " + "; ".join(report))
    assert not bad, "\n".join(bad)
    _assert_node_perturbation_caught(x1, x_dst, p, ref, g_out)


@pytest.mark.parametrize("mode", ["null_amax", "zero_grad", "tiny_2^-100", "huge_2^100"])
def test_node_backward_gradient_scale(mode):
    """grad_amax NULL (scale 1); an all-zero grad_out (every gradient exactly 0, never NaN); grad_out of max magnitude
    2^-100 and 2^100, held to the per-row bound of the unscaled case."""
    n_dst = 1000
    x1, x_dst, g_out = _node_inputs(n_dst, 43)
    p = _params(9)
    s = {"null_amax": 1.0, "zero_grad": 0.0, "tiny_2^-100": 2.0 ** -100, "huge_2^100": 2.0 ** 100}[mode]
    g = (g_out.double() * s).float() if s != 0 else torch.zeros_like(g_out)
    n_pn = 37
    _, _, g_x1, part = _node_launch(n_dst, x1, x_dst, p, g, n_pn, amax_mode="null" if mode == "null_amax" else "absmax")
    torch.cuda.synchronize()
    got = _unpack_node(part)
    if mode == "zero_grad":  # exact zeros: no tolerance to defend, the forward's perturbation check only
        assert bool((g_x1 == 0).all()), "grad_x1 of a zero grad_out must be exactly 0"
        for k, v in got.items():
            assert bool((v == 0).all()), f"grad {k} of a zero grad_out must be exactly 0"
        _assert_node_perturbation_caught(x1, x_dst, p, _node_reference(x1, x_dst, {k: v.to(D) for k, v in p.items()},
                                                                       None))
        return
    ref = _node_reference(x1, x_dst, {k: v.to(D) for k, v in p.items()}, g_out.double() * s)
    bad, report = [], []
    _check(bad, "grad_x1", g_x1, ref["grad"]["x_src"], TOL_GX1, report)
    for k, _, _ in NODE_SLICES:
        _check_weight(bad, f"grad {k}", got[k], ref["grad"][k], report)
    print(f"[node scale {mode}] " + "; ".join(report))
    assert not bad, "\n".join(bad)
    _assert_node_perturbation_caught(x1, x_dst, p, ref, g_out.double() * s)


def test_node_forward_accumulate_out_and_inference():
    """accumulate_out = 1 adds x_dst + MLP to what `out` holds (HeteroConv group "sum"); x2 = NULL (inference) gives the
    same `out` bit for bit."""
    n_dst = 2377
    x1, x_dst, _ = _node_inputs(n_dst, 47)
    p = _params(10)
    prev = torch.randn(n_dst, 16, 64, generator=torch.Generator().manual_seed(2)).cuda()
    out, x2, _, _ = _node_launch(n_dst, x1, x_dst, p, None, 1)
    out_inf, _, _, _ = _node_launch(n_dst, x1, x_dst, p, None, 1, with_x2=False)
    out_acc, _, _, _ = _node_launch(n_dst, x1, x_dst, p, None, 1, accumulate=prev)
    torch.cuda.synchronize()
    assert torch.equal(out, out_inf), "x2 = NULL changes out"
    ref = _node_reference(x1, x_dst, {k: v.to(D) for k, v in p.items()}, None)
    bad, report = [], []
    _check(bad, "out - x_dst", out - x_dst, ref["out"] - x_dst.to(D), TOL_OUT, report)
    _check(bad, "accumulated out - prev - x_dst", out_acc - prev - x_dst, ref["out"] - x_dst.to(D), TOL_OUT, report)
    print("[node accumulate] " + "; ".join(report))
    assert not bad, "\n".join(bad)
    # the kernel adds the old value to the residual first: the plain store with x_dst + prev as the residual
    out_sum, _, _, _ = _node_launch(n_dst, x1, x_dst + prev, p, None, 1)
    assert torch.equal(out_acc, out_sum), "accumulate_out is not out = (out + x_dst) + mlp"
    _assert_node_perturbation_caught(x1, x_dst, p, ref)


# ---------------------------------------------------------------------------------------------------------------------
# c-e. the whole fused layer
# ---------------------------------------------------------------------------------------------------------------------
LAYER_GRADS = ["x_src", "x_dst", "bw1", "bb1", "bw2", "bb2", "fk", "wk", "bias", "ln_g", "ln_b", "w1", "b1", "w2", "b2"]


def _fused_layer(es, x_src, x_dst, pos_src, pos_dst, p, dim, w, sub=None):
    """ops.fiber_conv with a BasisSpec on the 16-bit path: (out, {name: grad})."""
    from geometry_rl_b200 import ops
    leaves = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    xs = x_src.clone().requires_grad_(True)
    xd = None if x_dst is None else x_dst.clone().requires_grad_(True)
    ops.set_precision("bf16")
    try:
        basis = ops.BasisSpec(pos_src, pos_dst, leaves["bw1"], leaves["bb1"], leaves["bw2"], leaves["bb2"], _ori(dim), dim,
                              es)
        out = ops.fiber_conv(xs, xd, basis, leaves["fk"], leaves["wk"], leaves["bias"], leaves["ln_g"], leaves["ln_b"],
                             leaves["w1"], leaves["b1"], leaves["w2"], leaves["b2"], es, sub)
        out.backward(w)
    finally:
        ops.set_precision("fp32")
    grads = {k: v.grad for k, v in leaves.items()}
    grads["x_src"] = xs.grad
    if xd is not None:
        grads["x_dst"] = xd.grad
    return out.detach(), grads


def _compare_layer(tag, es, x_src, x_dst, pos_src, pos_dst, p, dim, w, sub=None, coo=None):
    out, grads = _fused_layer(es, x_src, x_dst, pos_src, pos_dst, p, dim, w, sub)
    torch.cuda.synchronize()
    ei = coo if coo is not None else es.coo
    kw = dict(x_src=x_src.to(D), x_dst=None if x_dst is None else x_dst.to(D), pos_src=pos_src.to(D),
              pos_dst=pos_dst.to(D), params={k: v.to(D) for k, v in p.items()}, ori3=_ori(dim).to(D), dim=dim,
              out_ids=None if sub is None else sub.out_ids, grad_out=w.to(D))
    ref = R.layer_reference(edge_index=ei, **kw)
    resid = (x_src if sub is None else x_src[sub.out_ids]) if x_dst is None else x_dst
    bad, report = [], []
    _check(bad, "out - x_dst", out - resid, ref["out"] - resid.to(D), TOL_OUT, report)
    for k in LAYER_GRADS:
        if k == "x_dst" and x_dst is None:
            continue
        if k == "x_dst":  # the residual's gradient is grad_out itself
            assert torch.equal(grads[k], w), "grad x_dst is not grad_out"
            continue
        if k == "x_src":
            _check(bad, "grad x_src", grads[k], ref["grad"][k], TOL_GXS, report)
        else:
            _check_weight(bad, f"grad {k}", grads[k], ref["grad"][k], report)
    print(f"[layer {tag}] " + "; ".join(report))
    assert not bad, "\n".join(bad)
    kw.pop("grad_out")
    if sub is not None:  # perturb one of the edges the sub layer reads
        ei = ei[:, torch.isin(ei[1], sub.out_ids)]
    pert = R.perturbed(R.layer_reference, ei, x_src.shape[0], **kw)
    for kind, res in pert.items():
        r = R.row_rel(res["out"] - resid.to(D), ref["out"] - resid.to(D))
        assert r >= 5 * TOL_OUT, f"{tag}: one {kind} edge moves out by only {r:.3e} < 5 x {TOL_OUT:g}"
    return out, grads


def _random_edge_set(B, ns, nd, e_per, seed, homo):
    from geometry_rl_b200 import ops
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(0, ns, (B, e_per), generator=g)
    dst = torch.randint(0, nd, (B, e_per), generator=g)
    if homo:
        src, dst = src.clamp_max(ns - 2), dst.clamp_max(nd - 2)  # a few nodes without edges
    coo = torch.stack([(src + (torch.arange(B) * ns)[:, None]).reshape(-1), (dst + (torch.arange(B) * nd)[:, None]).reshape(-1)])
    key = coo[0] * (B * nd) + coo[1]  # coalesced COO, like the data builders
    coo = coo[:, torch.sort(key).indices]
    return ops.build_edge_set(coo.cuda(), (torch.arange(B + 1) * e_per).cuda(), B, ns, nd)


def _layer_inputs(n_src, n_dst, n_out, seed, pos_scale=0.7):
    g = torch.Generator().manual_seed(seed)
    x_src = torch.randn(n_src, 16, 64, generator=g).cuda()
    x_dst = torch.randn(n_dst, 16, 64, generator=g).cuda()
    pos_src = (torch.randn(n_src, 3, generator=g) * pos_scale).cuda()
    pos_dst = (torch.randn(n_dst, 3, generator=g) * pos_scale).cuda()
    w = torch.randn(n_out, 16, 64, generator=g).cuda()
    return x_src, x_dst, pos_src, pos_dst, w


@pytest.mark.parametrize("kind", ["homogeneous", "bipartite", "sub"])
def test_fused_layer_against_fp64(kind):
    from geometry_rl_b200 import ops
    if kind == "bipartite":
        es = _random_edge_set(16, 30, 7, 90, 61, False)
        x_src, x_dst, pos_src, pos_dst, w = _layer_inputs(es.n_src, es.n_dst, es.n_dst, 62)
        _compare_layer(kind, es, x_src, x_dst, pos_src, pos_dst, _params(12), 3, w)
        return
    es = _random_edge_set(40, 49, 49, 128, 63, True)
    sub = ops.build_sub_edge_set(es, (torch.arange(40) * 49 + 3).cuda()) if kind == "sub" else None
    n_out = es.n_dst if sub is None else sub.n_dst
    x_src, _, pos_src, _, w = _layer_inputs(es.n_src, 1, n_out, 64)
    _compare_layer(kind, es, x_src, None, pos_src, pos_src, _params(13), 2, w, sub)


def test_fused_layer_on_a_capacity_radius_graph_with_an_empty_graph():
    """ops.radius_graph(..., capacity) with num_valid 0 for one graph of the batch (no edges there): the capacity set's
    tail entries point at node 0 and must not contribute."""
    from geometry_rl_b200 import ops
    B, P, r, m = 12, 40, 0.45, 6
    g = torch.Generator().manual_seed(71)
    pos = (torch.randn(B, P, 3, generator=g) * 0.5).cuda()
    nv = torch.tensor([40, 0, 33, 40, 17, 40, 40, 2, 40, 40, 39, 40], dtype=torch.int32).cuda()
    coo, ptr = ops.radius_graph(pos, nv, r, m, capacity=B * P * m)
    es = ops.build_edge_set(coo, ptr, B, P, P, exact=False)
    E = int(ptr[-1])
    assert E < B * P * m and int(ptr[2] - ptr[1]) == 0
    x_src, _, _, _, w = _layer_inputs(B * P, 1, B * P, 72)
    pos_f = pos.reshape(-1, 3).contiguous()
    _compare_layer("capacity radius", es, x_src, None, pos_f, pos_f, _params(14), 3, w, coo=coo[:, :E])


def test_fused_layer_bench_rope_topology():
    """The benchmark's rope workload at minibatch 2048 (kNN internal edges from the data builder); the fp64 reference of
    the whole layer with autograd fits in a few GB at this size."""
    t_name = "rope_shaping_hepi_trpl_cfg"
    from geometry_rl_b200.synthetic import CONFIGS, synthetic_obs
    cfg = CONFIGS[t_name]
    B = 2048
    obs = synthetic_obs(cfg, B, torch.Generator().manual_seed(23), env_ids=torch.arange(B) % cfg.num_envs)
    graph, _ = G.make_data(cfg, policy=True).build_data(*G.obs_args(cfg, obs, policy=True), train=False)
    es = graph.edge_sets[("links", "internal", "links")]
    pos = graph["links"].pos.float().contiguous()
    x_src, _, _, _, w = _layer_inputs(es.n_src, 1, es.n_dst, 73)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    _compare_layer(f"rope B={B}", es, x_src, None, pos, pos, _params(15), cfg.ponita_dim, w)
    print(f"[rope B={B}] {es.n_src} nodes, {es.n_edges} edges, peak device memory of the comparison "
          f"{(torch.cuda.max_memory_allocated() - base) / 2**30:.2f} GiB")


def _scale_case():
    es = _random_edge_set(24, 33, 33, 96, 81, True)
    x_src, _, pos, _, w = _layer_inputs(es.n_src, 1, es.n_dst, 82)
    return es, x_src, pos, w, _params(16)


def test_fused_layer_loss_scale_covariance():
    """Upstream gradient x 2^k, k in {-40, -20, 10, 20}: every gradient is exactly 2^k times the k = 0 gradient (the
    node backward's fp16 payload takes its scale from max|grad_out|, the edge backward's bf16 staging scales exactly).
    x 1e-7 and x 3e4 (not powers of two): within 2e-3 of each gradient's max after dividing for the node-side
    gradients; 1.5e-2 for the gradients of the edge backward (x_src, wk, basis MLP), whose bf16 staging of the kernel
    gradient rounds every value differently at another scale (measured 6.1e-3 for bb1 and 2.9e-3 for wk at 1e-7; their
    error against fp64 is up to 1.1e-2 at any scale)."""
    es, x_src, pos, w, p = _scale_case()
    _, base = _fused_layer(es, x_src, None, pos, pos, p, 3, w)
    for k in (-40, -20, 10, 20):
        _, gk = _fused_layer(es, x_src, None, pos, pos, p, 3, w * 2.0 ** k)
        for n, v in base.items():
            assert torch.equal(gk[n] / 2.0 ** k, v), f"grad {n} at 2^{k}: not exactly 2^{k} times the unscaled one"
    worst = {}
    for s in (1e-7, 3e4):
        _, gs = _fused_layer(es, x_src, None, pos, pos, p, 3, w * s)
        for n, v in base.items():
            worst[n] = max(worst.get(n, 0.0), R.global_rel(gs[n].double() / s, v))
    print("[loss scale] " + "; ".join(f"{n}: {e:.3e}" for n, e in worst.items()))
    for n, e in worst.items():
        assert e < (1.5e-2 if n in EDGE_SIDE else 2e-3), f"grad {n} at a non-power-of-two scale: {e:.2e}"


@pytest.mark.parametrize("case", ["long_edges", "small_weights"])
def test_fused_layer_dynamic_range(case):
    """Relative edge vectors up to 4x the longest edge of the synthetic observations (LONGEST_EDGE), and kernel.weight
    and the second basis-MLP weight at 2^-8 of their usual scale (the fibre kernel at 2^8, so that x2 keeps its scale):
    the same per-row bounds, finite outputs."""
    es = _random_edge_set(24, 33, 33, 96, 91, True)
    x_src, _, pos, _, w = _layer_inputs(es.n_src, 1, es.n_dst, 92)
    p = _params(17)
    if case == "long_edges":
        e = es.coo
        longest = float((pos[e[0]] - pos[e[1]]).norm(dim=1).max())
        pos = pos * (4 * LONGEST_EDGE / longest)
    else:
        p["wk"] = p["wk"] * 2.0 ** -8
        p["bw2"] = p["bw2"] * 2.0 ** -8
        p["fk"] = p["fk"] * 2.0 ** 8  # x2 keeps its scale, as the layer's one-time calibration of the fibre kernel does
    out, grads = _compare_layer(case, es, x_src, None, pos, pos, p, 3, w)
    assert bool(torch.isfinite(out).all()) and all(bool(torch.isfinite(v).all()) for v in grads.values())
