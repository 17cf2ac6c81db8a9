"""GPU: the strict fp32 convolution kernels and the one-time calibration alone against fp64 references
(tests/conv16_reference.py, tests/conv32_reference.py), with a per-row metric, at tile, block and grid-stride edges.

a. grl_edge_basis_fwd / _bwd through the C ABI: the basis [E,16,64] row by row, the four basis-MLP weight gradients;
   E around the 8-edge tile and the forward's 3 x SMs grid-stride, both dims, edges up to 4 x LONGEST_EDGE, coincident
   endpoints; every partial count, idle slots exactly zero;
b. grl_fbconv_edge_fwd / _bwd through the C ABI, fed a random basis: x1, grad_x_src, grad_basis, grad wk; hubs of
   degree 5000, degrees 0..17 on both sides, empty 16-node blocks, n_dst around the forward's 2 x SMs grid, no edges,
   one source, bipartite sets and the data builders' topologies; grad_x_src_init null and set, accumulate_grad_basis,
   sub-layer addressing through the parent's arrays, every partial count, repeatability;
c. grl_fbconv_node_fwd / _bwd through the C ABI, fed a random x1: out - x_dst, grad_x1 and the eight node gradients
   around the 8-node tile and the 2 x SMs grid, every partial count, accumulate_out, and the LayerNorm rows the model
   produces (constant rows, a large common offset, x1 at 1e-3 and 1e3);
d. the whole strict layer, ops.fiber_conv on a materialised fp32 basis (EdgeBasisFn): homogeneous, bipartite, sub
   layer, two layers sharing one basis, the HEPi and EMPN builders' topologies with the pruned sub set;
e. the one-time calibration: ops.aggregate_messages in both precisions, the factors of conv.py and ponita.py against
   fp64, a capacity radius set, and the module's first and second training forward.

Every output and partial buffer is filled with NaN before a launch; grids are sized from _lib.sm_count() at run time.
Exact properties (zero rows, init rows, repeatability, bit-identity across partial counts) use torch.equal.  Every case
shows that its own per-row tolerance puts one dropped edge or one swapped source (conv16_reference.perturbed) at 5x or
more of it.

Error model and tolerances.  The strict kernels are fp32 FFMA with erf GELU, the same operator as the reference, so
their error is fp32 rounding: about 2^-24 times the magnitude of the terms each output sums.  A per-row error
(conv16_reference.row_rel, floor 1% of the tensor's max) of a 64-term contraction sits near 1e-6.  A segmented sum over
`deg` edges adds its messages one after the other in one thread; with messages of independent signs its rounding error
grows like sqrt(deg), so a row of x1 (grad_x_src) is held to TOL * sqrt(max(1, deg / 16)) with `deg` the largest
in-degree (out-degree) of the case (_deg_tol): the 5000-edge hubs are held to 17.7 x TOL (measured 2.7e-6 for x1 and
4.6e-6 for grad_x_src there, the same order as degree 16).  A LayerNorm row whose values share an offset `m` much
larger than their spread `s` loses m/s * 2^-24 in x2 itself (the fp32 value of x2 rounds at the offset's scale), so
that case is held to TOL + m/s * OFFSET_ULPS * 2^-24 (m/s up to 256 there: measured 2.8e-5 for out, 2.0e-5 for grad_x1,
1.4e-5 for grad w2).  Weight gradients sum over every edge or node: global max-norm bounds.  Worst cases measured on
one B200 (1000 W power limit) over every case of this file are recorded next to each bound; every whole-layer error is
below 1.3e-6, under north_star's 1e-5.  The file runs in about 15 s on one B200."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from tests import conv16_reference as R
from tests import conv32_reference as R32
from tests import gpu_helpers as G
from tests.conv16_reference import LONGEST_EDGE, random_params

pytestmark = pytest.mark.gpu

D = torch.float64
NAN = float("nan")
U = 2.0 ** -24
# per-row (row_rel, floor 1e-2) bounds of the strict kernels, measured worst case (case)
TOL_BASIS = 4e-6      # basis rows of grl_edge_basis_fwd: 9.5e-7 (200003 edges, dim 3)
TOL_X1 = 4e-6         # x1 rows of grl_fbconv_edge_fwd at degree <= 16: 9.4e-7 (one source)
TOL_GXS = 4e-6        # grad_x_src rows of grl_fbconv_edge_bwd at degree <= 16: 8.7e-7 (rope kNN); 1.1e-6 at degree 310
TOL_GB = 4e-6         # grad_basis rows of grl_fbconv_edge_bwd: 8.7e-7 (rigid TASK edges)
TOL_OUT = 6e-6        # out - x_dst rows of grl_fbconv_node_fwd: 1.7e-6 (n_dst 20011)
TOL_GX1 = 6e-6        # grad_x1 rows of grl_fbconv_node_bwd: 1.5e-6 (n_dst 20011)
OFFSET_ULPS = 4       # offset term of a LayerNorm row: TOL + m/s * OFFSET_ULPS * 2^-24
# global max-norm bound of the weight gradients at the partial counts of EdgeBasisFn / FiberConvFn: 1.4e-5 (grad w2,
# LayerNorm offset rows), 1.1e-5 (grad wk, a source of out-degree 5000: one CTA sums its 5000 edges)
GLOBAL_W = 5e-5
# any other partial count, against the default count and against fp64: n_partials = 1 makes one CTA sum every tile in
# fp32 (25000 tiles of 128 rows for 200003 edges), which moves the basis-MLP gradients by up to 6.9e-5 of their max
REASSOC = 2e-4
# north_star's bound of the strict path, whole layer, output and every gradient (worst 1.3e-6, grad bb2, HEPi internal)
NORTH_STAR = 1e-5
# 16-bit bounds of the calibration input in bf16 mode (the materialised bf16 basis of grl_edge_basis_fwd_tc):
TOL_BASIS16 = 2e-2    # measured 8.0e-3
TOL_X1_16 = 3e-2      # measured 1.4e-2

_ORI = {}


def _ori(dim):
    if dim not in _ORI:
        from geometry_rl_b200.modules.pyg_models.ponita.ponita import make_ori_grid, pad_ori3
        _ORI[dim] = pad_ori3(make_ori_grid(dim, 16, False).cuda()).contiguous()
    return _ORI[dim]


def _params(seed, **kw):
    return {k: v.cuda() for k, v in random_params(torch.Generator().manual_seed(seed), torch.float32, **kw).items()}


def _sms():
    from geometry_rl_b200 import _lib as L
    return L.sm_count()


def _deg_tol(tol, deg):
    return tol * max(1.0, (deg / 16) ** 0.5)


def _row(bad, report, name, got, ref, tol):
    r, g = R.row_rel(got, ref), R.global_rel(got, ref)
    report.append(f"{name}: row {r:.3e} (tol {tol:.2e}) global {g:.3e}")
    if not r < tol:
        bad.append(f"{name}: row {r:.3e} > tol {tol:.2e}")
    return r


def _glob(bad, report, name, got, ref, tol=GLOBAL_W):
    g = R.global_rel(got, ref)
    report.append(f"{name}: global {g:.3e} (tol {tol:.0e})")
    if not g < tol:
        bad.append(f"{name}: global {g:.3e} > tol {tol:.0e}")
    return g


def _finish(tag, bad, report):
    print(f"[{tag}] " + "; ".join(report))
    assert not bad, f"{tag}:\n" + "\n".join(bad)


# ---------------------------------------------------------------------------------------------------------------------
# a. edge basis alone
# ---------------------------------------------------------------------------------------------------------------------
def _basis_pack(p):
    """The operands of grl_edge_basis_* as EdgeBasisFn fills them: w1t [16,64] zero-padded, w2t = w2^T, w2."""
    w1t = torch.zeros(16, 64, device="cuda")
    w1t[:14] = p["bw1"].t()
    return dict(w1t=w1t.contiguous(), w2t=p["bw2"].t().contiguous(), w2=p["bw2"].contiguous())


def _basis_desc(E, dim, e_src, e_dst, pos_src, pos_dst, p, pk, **kw):
    from geometry_rl_b200 import _lib as L
    return L.GrlBasisDesc(n_edges=E, dim=dim, edge_src=L.ptr(e_src), edge_dst=L.ptr(e_dst), pos_src=L.ptr(pos_src),
                          pos_dst=L.ptr(pos_dst), ori=L.ptr(_ori(dim)), w1t=L.ptr(pk["w1t"]), b1=L.ptr(p["bb1"]),
                          w2t=L.ptr(pk["w2t"]), b2=L.ptr(p["bb2"]), w2=L.ptr(pk["w2"]),
                          **{k: L.ptr(v) if isinstance(v, torch.Tensor) else v for k, v in kw.items()})


def _basis_fwd(E, dim, e_src, e_dst, pos_src, pos_dst, p, pk):
    from geometry_rl_b200 import _lib as L
    basis = torch.full((E, 16, 64), NAN, device="cuda")
    L.call("grl_edge_basis_fwd", C.byref(_basis_desc(E, dim, e_src, e_dst, pos_src, pos_dst, p, pk, basis=basis)))
    return basis


def _basis_bwd(E, dim, e_src, e_dst, pos_src, pos_dst, p, pk, g_basis, n_p):
    from geometry_rl_b200 import _lib as L
    part = torch.full((n_p, L.BASIS_GRAD_FLOATS), NAN, device="cuda")
    L.call("grl_edge_basis_bwd", C.byref(_basis_desc(E, dim, e_src, e_dst, pos_src, pos_dst, p, pk, grad_basis=g_basis,
                                                     grad_partials=part, n_partials=n_p)))
    return part


def _unpack_basis(part):
    g = part.double().sum(0)
    w1 = g[:1024].view(64, 16)
    return {"bw1": w1[:, :14], "bb1": g[1024:1088], "bw2": g[1088:5184].view(64, 64), "bb2": g[5184:]}, w1[:, 14:]


def _basis_count(name):
    s = _sms()
    return {"1": 1, "7": 7, "8": 8, "9": 9, "24G-1": 24 * s - 1, "24G+9": 24 * s + 9, "200k": 200003}[name]


def _basis_case(E, seed, longest=None):
    """E edges between n_src sources and n_dst destinations at positions ~N(0, 0.6); every 7th edge (from the 4th) has
    coincident endpoints (its destination sits at its source's position).  `longest`: scale so that the longest edge
    has that length."""
    g = torch.Generator().manual_seed(seed)
    n_src, n_plain = max(2, E // 3), max(1, E // 3)
    src = torch.randint(0, n_src, (E,), generator=g)
    dst = torch.randint(0, n_plain, (E,), generator=g)
    pos_src = torch.randn(n_src, 3, generator=g) * 0.6
    pos_dst = torch.randn(n_plain, 3, generator=g) * 0.6
    co = torch.arange(3, max(E, 3), 7)
    dst[co] = n_plain + torch.arange(co.numel())
    pos_dst = torch.cat([pos_dst, pos_src[src[co]]])
    if longest is not None:
        s = longest / float((pos_src[src] - pos_dst[dst]).norm(dim=1).max())
        pos_src, pos_dst = pos_src * s, pos_dst * s
    return src, dst, pos_src, pos_dst


BASIS_COUNTS = ["1", "7", "8", "9", "24G-1", "24G+9", "200k"]
BASIS_CASES = [(n, d, "typical") for n in BASIS_COUNTS for d in (2, 3)] + [("24G+9", 2, "long"), ("24G+9", 3, "long")]


@pytest.mark.parametrize("count,dim,geom", BASIS_CASES, ids=[f"E{n}-dim{d}-{g}" for n, d, g in BASIS_CASES])
def test_edge_basis_kernels_alone_against_fp64(count, dim, geom):
    E = _basis_count(count)
    src, dst, pos_src, pos_dst = _basis_case(E, 100 + E + dim, 4 * LONGEST_EDGE if geom == "long" else None)
    e_src, e_dst = src.int().cuda(), dst.int().cuda()
    pos_src, pos_dst = pos_src.cuda(), pos_dst.cuda()
    p = _params(20 + dim)
    pk = _basis_pack(p)
    g_basis = torch.randn(E, 16, 64, generator=torch.Generator().manual_seed(E)).cuda()
    n_tiles = (E + 7) // 8
    n_p0 = max(1, min(n_tiles, _sms()))  # EdgeBasisFn's count in fp32 mode

    basis = _basis_fwd(E, dim, e_src, e_dst, pos_src, pos_dst, p, pk)
    part = _basis_bwd(E, dim, e_src, e_dst, pos_src, pos_dst, p, pk, g_basis, n_p0)
    torch.cuda.synchronize()
    ei = torch.stack([src, dst]).cuda()
    kw = dict(pos_src=pos_src.to(D), pos_dst=pos_dst.to(D), params=p, ori3=_ori(dim).to(D), dim=dim)
    ref = R32.basis_reference(edge_index=ei, grad_basis=g_basis.to(D), **kw)
    bad, report = [], []
    _row(bad, report, "basis", basis, ref["basis"], TOL_BASIS)
    got, pad = _unpack_basis(part)
    for k in R32.BASIS:
        _glob(bad, report, f"grad {k}", got[k], ref["grad"][k])
    assert bool((pad == 0).all()), "gradient of the zero-padded feature columns 14, 15 is not 0"

    # exact: a second launch gives the same bits
    assert torch.equal(basis, _basis_fwd(E, dim, e_src, e_dst, pos_src, pos_dst, p, pk)), "forward not repeatable"
    assert torch.equal(part, _basis_bwd(E, dim, e_src, e_dst, pos_src, pos_dst, p, pk, g_basis, n_p0)), \
        "backward not repeatable"
    # every partial count: fp32 reassociation of the per-CTA sums only; slots of CTAs without a tile are exactly 0
    worst = 0.0
    for n_p in sorted({1, 7, n_tiles, n_tiles + 3}):
        pp = _basis_bwd(E, dim, e_src, e_dst, pos_src, pos_dst, p, pk, g_basis, n_p)
        gp, _ = _unpack_basis(pp)
        for k in R32.BASIS:
            worst = max(worst, R.global_rel(gp[k], got[k]))
            _glob(bad, [], f"n_partials={n_p} grad {k}", gp[k], ref["grad"][k], REASSOC)
        if n_p > n_tiles:
            assert torch.equal(pp[n_tiles:], torch.zeros_like(pp[n_tiles:])), f"n_partials={n_p}: idle slot not 0"
    report.append(f"partial counts: reassociation {worst:.3e} (tol {REASSOC:.0e})")
    if not worst < REASSOC:
        bad.append(f"partial counts move the gradients by {worst:.3e}")
    _finish(f"basis E={E} dim={dim} {geom}", bad, report)

    # the tolerance catches one edge with a swapped source (the last edge, in the last, possibly partial tile)
    sw = ei.clone()
    sw[0, E - 1] = (sw[0, E - 1] + 1) % pos_src.shape[0]
    r = R.row_rel(R32.basis_reference(edge_index=sw, **kw)["basis"], ref["basis"])
    assert r >= 5 * TOL_BASIS, f"one swapped source moves the basis by {r:.3e} only"


# ---------------------------------------------------------------------------------------------------------------------
# b. spatial half alone
# ---------------------------------------------------------------------------------------------------------------------
class Topo:
    """An edge list in the layouts of ops.EdgeSet: edge order (dst-sorted, ties in COO order) with rowptr_dst, and the
    src-sorted walk (ties in edge order) as src_eid with rowptr_src; `ei` [3,E] = (src, dst, edge-order position)."""

    def __init__(self, src, dst, n_src, n_dst):
        src, dst = src.long().cuda(), dst.long().cuda()
        o = torch.sort(dst, stable=True).indices
        self.edge_src, self.edge_dst = src[o].int().contiguous(), dst[o].int().contiguous()
        self.src_eid = torch.sort(self.edge_src.long(), stable=True).indices.int().contiguous()
        self.rowptr_dst = self._rowptr(self.edge_dst, n_dst)
        self.rowptr_src = self._rowptr(self.edge_src, n_src)
        self.n_src, self.n_dst, self.n_edges = n_src, n_dst, int(src.numel())
        self.ei = torch.stack([self.edge_src.long(), self.edge_dst.long(), torch.arange(self.n_edges, device="cuda")])

    @staticmethod
    def _rowptr(keys, n):
        rp = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
        rp[1:] = torch.cumsum(torch.bincount(keys.long(), minlength=n), 0)
        return rp.int().contiguous()

    @classmethod
    def of_edge_set(cls, es):
        return cls(es.edge_src, es.edge_dst, es.n_src, es.n_dst)


def _edge_pack(wk):
    return wk.t().contiguous(), wk.contiguous()


def _spatial_fwd(n_src, n_dst, n_edges, rowptr_dst, edge_src, edge_dst, x_src, basis, wk):
    from geometry_rl_b200 import _lib as L
    x1 = torch.full((n_dst, 16, 64), NAN, device="cuda")
    wk_t, _ = _edge_pack(wk)
    d = L.GrlConvDesc(n_src=n_src, n_dst=n_dst, n_edges=n_edges, rowptr_dst=L.ptr(rowptr_dst), edge_src=L.ptr(edge_src),
                      edge_dst=L.ptr(edge_dst), x_src=L.ptr(x_src), basis=L.ptr(basis), wk_t=L.ptr(wk_t), x1=L.ptr(x1))
    L.call("grl_fbconv_edge_fwd", C.byref(d))
    return x1


def _spatial_bwd(n_src, n_dst, n_edges, rowptr_src, src_eid, edge_src, edge_dst, x_src, basis, wk, g_x1, n_p,
                 init=None, g_basis=None, accumulate=0):
    """grad_x_src (NaN-filled), grad_basis (NaN-filled unless `g_basis` is given: then written into a copy of it) and
    the partial slots."""
    from geometry_rl_b200 import _lib as L
    g_xs = torch.full((n_src, 16, 64), NAN, device="cuda")
    if g_basis is None:
        g_basis = torch.full((max(n_edges, 1), 16, 64), NAN, device="cuda") if basis is not None else None
    else:
        g_basis = g_basis.clone()
    part = torch.full((n_p, L.EDGE_GRAD_FLOATS), NAN, device="cuda")
    wk_t, wk_c = _edge_pack(wk)
    d = L.GrlConvDesc(n_src=n_src, n_dst=n_dst, n_edges=n_edges, rowptr_src=L.ptr(rowptr_src), src_eid=L.ptr(src_eid),
                      edge_src=L.ptr(edge_src), edge_dst=L.ptr(edge_dst), x_src=L.ptr(x_src), basis=L.ptr(basis),
                      wk_t=L.ptr(wk_t), wk=L.ptr(wk_c), grad_x1=L.ptr(g_x1), grad_x_src=L.ptr(g_xs),
                      grad_x_src_init=L.ptr(init), grad_basis=L.ptr(g_basis), accumulate_grad_basis=accumulate,
                      edge_grad_partials=L.ptr(part), n_partials_edge=n_p)
    L.call("grl_fbconv_edge_bwd", C.byref(d))
    return g_xs, g_basis, part


def _fwd(t, x_src, basis, wk):
    return _spatial_fwd(t.n_src, t.n_dst, t.n_edges, t.rowptr_dst, t.edge_src, t.edge_dst, x_src, basis, wk)


def _bwd(t, x_src, basis, wk, g_x1, n_p, **kw):
    return _spatial_bwd(t.n_src, t.n_dst, t.n_edges, t.rowptr_src, t.src_eid, t.edge_src, t.edge_dst, x_src, basis, wk,
                        g_x1, n_p, **kw)


def _spatial_ref(edge_index, basis, **kw):
    """spatial_reference over a [3,E] edge list whose row 2 is the basis row of every edge (so that a perturbed list
    keeps every other edge's basis)."""
    return R32.spatial_reference(basis=basis[edge_index[2]], edge_index=edge_index[:2], **kw)


def _spatial_case(name):
    """(src, dst, n_src, n_dst)."""
    s = _sms()
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    ri = lambda hi, n: torch.randint(0, hi, (n,), generator=g)  # noqa: E731
    if name == "hub_dst":  # one destination of in-degree 5000 (one thread's sequential sum over 625 tiles)
        src = torch.cat([torch.arange(5000), torch.tensor([0, 1, 2, 3, 4])])
        dst = torch.cat([torch.zeros(5000, dtype=torch.long), torch.tensor([1, 1, 2, 2, 2])])
        return src, dst, 5002, 4
    if name == "hub_src":  # one source of out-degree 5000 (the backward's key side)
        src = torch.cat([torch.zeros(5000, dtype=torch.long), torch.tensor([1, 1, 2])])
        dst = torch.cat([torch.arange(5000), torch.tensor([0, 7, 7])])
        return src, dst, 4, 5002
    if name == "mod8":  # per-node degrees 0, 1, 7, 8, 9, 15, 16, 17 on both sides
        degs = torch.tensor([8, 9, 15, 0, 1, 7, 16, 17, 2] * 6)
        dst = torch.repeat_interleave(torch.arange(degs.numel()), degs)
        src = torch.repeat_interleave(torch.arange(degs.numel()), degs.roll(4))[torch.randperm(dst.numel(), generator=g)]
        return src, dst, degs.numel(), degs.numel()
    if name == "empty_blocks":  # 16-node blocks 0, 2, 3 and 7.. without edges on both sides, trailing nodes after the last
        live = torch.cat([torch.arange(16, 32), torch.arange(64, 100)])
        dst = live[ri(live.numel(), 400)]
        src = live[ri(live.numel(), 400)]
        return src, dst, 16 * 9 + 5, 16 * 9 + 5
    if name.startswith("n_dst="):  # n_dst around the forward's grid (2 x SMs blocks of 16): every block, grid strides
        n = {"1": 1, "15": 15, "16": 16, "17": 17, "32G-16": 32 * s - 16, "32G+16": 32 * s + 16}[name[6:]]
        n_src = max(2, n // 2 + 3)
        E = 2 * n + 3
        return ri(n_src, E), ri(n, E), n_src, n
    if name == "one_src":  # n_src = 1
        dst = torch.cat([torch.arange(300), torch.arange(10)])
        return torch.zeros(dst.numel(), dtype=torch.long), dst, 1, 301
    if name == "bipartite":
        return ri(700, 4000), ri(300, 4000), 703, 300
    raise KeyError(name)


def _builder_topology(kind):
    """Edge sets the data builders make: rope kNN internal edges at minibatch 64, rigid TASK edges at minibatch 1024."""
    from geometry_rl_b200.synthetic import CONFIGS, synthetic_obs
    name = "rope_shaping_hepi_trpl_cfg" if kind == "rope_knn" else "rigid_insertion_multi_hepi_trpl_cfg"
    cfg = CONFIGS[name]
    B = 64 if kind == "rope_knn" else 1024
    obs = synthetic_obs(cfg, B, torch.Generator().manual_seed(21), env_ids=torch.arange(B) % cfg.num_envs)
    graph, _ = G.make_data(cfg, policy=True).build_data(*G.obs_args(cfg, obs, policy=True), train=False)
    et = ("links", "internal", "links") if kind == "rope_knn" else ("object_geometry", "task", "grippers")
    from geometry_rl_b200 import ops
    return Topo.of_edge_set(ops.exact_edge_set(graph.edge_sets[et]))


SPATIAL_CASES = ["hub_dst", "hub_src", "mod8", "empty_blocks", "n_dst=1", "n_dst=15", "n_dst=16", "n_dst=17",
                 "n_dst=32G-16", "n_dst=32G+16", "one_src", "bipartite", "rope_knn", "rigid_task"]


def _spatial_inputs(t, seed=17):
    g = torch.Generator().manual_seed(seed)
    x_src = torch.randn(t.n_src, 16, 64, generator=g).cuda()
    basis = (torch.randn(max(t.n_edges, 1), 16, 64, generator=g) * 0.5).cuda()
    g_x1 = torch.randn(t.n_dst, 16, 64, generator=g).cuda()
    init = torch.randn(t.n_src, 16, 64, generator=g).cuda()
    g0 = torch.randn(max(t.n_edges, 1), 16, 64, generator=g).cuda()
    return x_src, basis, g_x1, init, g0


@pytest.mark.parametrize("name", SPATIAL_CASES)
def test_spatial_kernels_alone_against_fp64(name):
    if name in ("rope_knn", "rigid_task"):
        t = _builder_topology(name)
    else:
        t = Topo(*_spatial_case(name))
    x_src, basis, g_x1, init, g0 = _spatial_inputs(t)
    wk = _params(3)["wk"]
    n_blocks = (t.n_src + 15) // 16
    n_p0 = max(1, min(n_blocks, _sms()))  # FiberConvFn's count in fp32 mode
    use_init = init if t.n_src % 2 == 0 else None

    x1 = _fwd(t, x_src, basis, wk)
    g_xs, g_b, part = _bwd(t, x_src, basis, wk, g_x1, n_p0, init=use_init)
    torch.cuda.synchronize()
    kw = dict(x_src=x_src.to(D), wk=wk.to(D), n_dst=t.n_dst, grad_x1=g_x1.to(D))
    ref = _spatial_ref(t.ei, basis.to(D), **kw)
    ref_gxs = ref["grad"]["x_src"] + (init.to(D) if use_init is not None else 0)
    deg_in = (t.rowptr_dst[1:] - t.rowptr_dst[:-1]).long()
    deg_out = (t.rowptr_src[1:] - t.rowptr_src[:-1]).long()
    tol_x1, tol_gxs = _deg_tol(TOL_X1, int(deg_in.max())), _deg_tol(TOL_GXS, int(deg_out.max()))
    bad, report = [], [f"{t.n_src} src, {t.n_dst} dst, {t.n_edges} edges, max degree in {int(deg_in.max())} "
                        f"out {int(deg_out.max())}"]
    _row(bad, report, "x1", x1, ref["x1"], tol_x1)
    _row(bad, report, "grad_x_src", g_xs, ref_gxs, tol_gxs)
    _row(bad, report, "grad_basis", g_b, ref["grad"]["basis"], TOL_GB)
    _glob(bad, report, "grad wk", part.double().sum(0).view(64, 64), ref["grad"]["wk"])

    # exact: rows without an edge (the forward's zero-fill path; the backward's init-only path)
    assert torch.equal(x1[deg_in == 0], torch.zeros_like(x1[deg_in == 0])), "x1 of a node without in-edges is not 0"
    want = init[deg_out == 0] if use_init is not None else torch.zeros_like(g_xs[deg_out == 0])
    assert torch.equal(g_xs[deg_out == 0], want), "grad_x_src of a source without out-edges is not its init (or 0)"
    # exact: init set vs null is one fp32 add per element; accumulate_grad_basis = 1 adds to what the buffer held
    g_xs_other, g_b_acc, _ = _bwd(t, x_src, basis, wk, g_x1, n_p0, init=None if use_init is not None else init,
                                  g_basis=g0, accumulate=1)
    with_init, without = (g_xs, g_xs_other) if use_init is not None else (g_xs_other, g_xs)
    assert torch.equal(with_init, without + init), "grad_x_src with an init is not (the sum without it) + init"
    assert torch.equal(g_b_acc, g_b + g0), "accumulate_grad_basis = 1 does not add to the buffer"
    # exact: a second launch gives the same bits
    x1b = _fwd(t, x_src, basis, wk)
    g_xsb, g_bb, partb = _bwd(t, x_src, basis, wk, g_x1, n_p0, init=use_init)
    assert torch.equal(x1, x1b) and torch.equal(g_xs, g_xsb) and torch.equal(g_b, g_bb) and torch.equal(part, partb), \
        "not repeatable"
    # every partial count: the same grad_x_src / grad_basis bits, grad wk up to reassociation, idle slots 0
    worst = 0.0
    for n_p in sorted({1, 7, n_blocks, n_blocks + 3}):
        g_xs2, g_b2, part2 = _bwd(t, x_src, basis, wk, g_x1, n_p, init=use_init)
        assert torch.equal(g_xs2, g_xs) and torch.equal(g_b2, g_b), f"grad_x_src / grad_basis depend on n_partials={n_p}"
        worst = max(worst, R.global_rel(part2.double().sum(0), part.double().sum(0)))
        if n_p > n_blocks:
            assert torch.equal(part2[n_blocks:], torch.zeros_like(part2[n_blocks:])), f"n_partials={n_p}: idle slot not 0"
    report.append(f"partial counts: reassociation {worst:.3e} (tol {REASSOC:.0e})")
    if not worst < REASSOC:
        bad.append(f"partial counts move grad wk by {worst:.3e}")
    _finish(f"spatial {name}", bad, report)

    # the tolerance catches one dropped / one misrouted edge (x1 or grad_x_src, whichever the topology lets one edge
    # dominate a row of)
    for kind in (("drop", "swap") if t.n_src >= 2 else ("drop",)):
        pe = _spatial_ref(R.perturbation(t.ei, kind, t.n_src), basis.to(D), **kw)
        pg = pe["grad"]["x_src"] + (init.to(D) if use_init is not None else 0)
        r1, r2 = R.row_rel(pe["x1"], ref["x1"]), R.row_rel(pg, ref_gxs)
        assert max(r1 / tol_x1, r2 / tol_gxs) >= 5, f"one {kind} edge: x1 {r1:.3e}, grad_x_src {r2:.3e}"


def test_spatial_kernels_without_edges():
    """n_edges = 0 with a null basis and null grad_basis: x1 exactly 0, grad_x_src exactly the init (or 0), every
    partial slot exactly 0."""
    t = Topo(torch.zeros(0, dtype=torch.long), torch.zeros(0, dtype=torch.long), 37, 21)
    x_src, _, g_x1, init, _ = _spatial_inputs(t)
    wk = _params(3)["wk"]
    x1 = _fwd(t, x_src, None, wk)
    for use_init in (None, init):
        for n_p in (1, 3, 5):
            g_xs, _, part = _bwd(t, x_src, None, wk, g_x1, n_p, init=use_init)
            assert torch.equal(g_xs, init if use_init is not None else torch.zeros_like(g_xs))
            assert torch.equal(part, torch.zeros_like(part))
    assert torch.equal(x1, torch.zeros_like(x1))


def test_spatial_kernels_sub_layer_addressing():
    """A sub layer as FiberConvFn runs it (the last EMPN layer): the forward over the subset's own arrays and a compact
    basis copy; the backward through the PARENT's edge_src, edge_dst_parent ranks, src_eid_parent, basis and a
    parent-sized grad_basis.  Rows of grad_basis outside the subset keep their bits, with and without accumulation."""
    from geometry_rl_b200 import ops
    B, n, e_per = 24, 37, 100
    g = torch.Generator().manual_seed(51)
    src = torch.randint(0, n - 2, (B, e_per), generator=g)
    dst = torch.randint(0, n - 2, (B, e_per), generator=g)
    off = (torch.arange(B) * n)[:, None]
    coo = torch.stack([(src + off).reshape(-1), (dst + off).reshape(-1)])
    coo = coo[:, torch.sort(coo[0] * (B * n) + coo[1]).indices]
    es = ops.build_edge_set(coo.cuda(), (torch.arange(B + 1) * e_per).cuda(), B, n, n)
    sub = ops.build_sub_edge_set(es, (torch.arange(B) * n + 5).cuda())
    x_src, basis, _, _, sentinel = _spatial_inputs(Topo.of_edge_set(es), 53)
    g_x1 = torch.randn(sub.n_dst, 16, 64, generator=g).cuda()
    wk = _params(4)["wk"]
    n_p = max(1, min((es.n_src + 15) // 16, _sms()))
    x1 = _spatial_fwd(es.n_src, sub.n_dst, sub.n_edges, sub.rowptr_dst, sub.edge_src, sub.edge_dst, x_src,
                      basis.index_select(0, sub.eids), wk)
    args = (es.n_src, sub.n_dst, sub.n_edges, sub.rowptr_src, sub.src_eid_parent, es.edge_src, sub.edge_dst_parent,
            x_src, basis, wk, g_x1, n_p)
    g_xs, g_b, part = _spatial_bwd(*args, g_basis=sentinel)
    _, g_b_acc, _ = _spatial_bwd(*args, g_basis=sentinel, accumulate=1)
    torch.cuda.synchronize()
    ei = torch.stack([sub.edge_src.long(), sub.edge_dst.long(), sub.eids])
    ref = _spatial_ref(ei, basis.to(D), x_src=x_src.to(D), wk=wk.to(D), n_dst=sub.n_dst, grad_x1=g_x1.to(D))
    # the reference's basis gradient is per sub-edge; scatter it to the parent rows
    ref_gb = torch.zeros(es.n_edges, 16, 64, dtype=D, device="cuda").index_add_(0, sub.eids, ref["grad"]["basis"])
    inside = torch.zeros(es.n_edges, dtype=torch.bool, device="cuda")
    inside[sub.eids] = True
    bad, report = [], [f"{sub.n_edges} of {es.n_edges} edges"]
    _row(bad, report, "x1", x1, ref["x1"], _deg_tol(TOL_X1, int((sub.rowptr_dst[1:] - sub.rowptr_dst[:-1]).max())))
    _row(bad, report, "grad_x_src", g_xs, ref["grad"]["x_src"],
         _deg_tol(TOL_GXS, int((sub.rowptr_src[1:] - sub.rowptr_src[:-1]).max())))
    _row(bad, report, "grad_basis (subset rows)", g_b[inside], ref_gb[inside], TOL_GB)
    _glob(bad, report, "grad wk", part.double().sum(0).view(64, 64), ref["grad"]["wk"])
    _finish("spatial sub layer", bad, report)
    assert torch.equal(g_b[~inside], sentinel[~inside]), "grad_basis rows outside the subset were written"
    assert torch.equal(g_b_acc[~inside], sentinel[~inside]), "grad_basis rows outside the subset were written (accumulate)"
    assert torch.equal(g_b_acc[inside], g_b[inside] + sentinel[inside]), "accumulate_grad_basis does not add"
    pe = _spatial_ref(R.perturbation(ei, "drop", es.n_src), basis.to(D), x_src=x_src.to(D), wk=wk.to(D), n_dst=sub.n_dst)
    assert R.row_rel(pe["x1"], ref["x1"]) >= 5 * TOL_X1


# ---------------------------------------------------------------------------------------------------------------------
# c. node half alone
# ---------------------------------------------------------------------------------------------------------------------
def _node_pack(p):
    """w1_t, w2_t, w2_c as FiberConvFn fills them for the strict kernels."""
    w1, w2 = p["w1"], p["w2"]
    return dict(w1_t=w1.view(4, 64, 64).transpose(1, 2).contiguous(), w1=w1.contiguous(),
                w2_t=w2.view(64, 4, 64).permute(1, 2, 0).contiguous(), w2_c=w2.view(64, 4, 64).permute(1, 0, 2).contiguous())


def _node_launch(x1, x_dst, p, g_out, n_pn, accumulate=None):
    from geometry_rl_b200 import _lib as L
    n = x1.shape[0]
    pk = _node_pack(p)
    out = torch.full((n, 16, 64), NAN, device="cuda") if accumulate is None else accumulate.clone()
    d = L.GrlConvDesc(n_src=n, n_dst=n, n_edges=0, x_dst=L.ptr(x_dst), fiber_kernel=L.ptr(p["fk"]), bias=L.ptr(p["bias"]),
                      ln_g=L.ptr(p["ln_g"]), ln_b=L.ptr(p["ln_b"]), w1_t=L.ptr(pk["w1_t"]), w1=L.ptr(pk["w1"]),
                      b1=L.ptr(p["b1"]), w2_t=L.ptr(pk["w2_t"]), w2_c=L.ptr(pk["w2_c"]), b2=L.ptr(p["b2"]), x1=L.ptr(x1),
                      out=L.ptr(out), accumulate_out=int(accumulate is not None))
    L.call("grl_fbconv_node_fwd", C.byref(d))
    if g_out is None:
        return out, None, None
    g_x1 = torch.full_like(x1, NAN)
    part = torch.full((n_pn, L.NODE_GRAD_FLOATS), NAN, device="cuda")
    d.grad_out, d.grad_x1, d.node_grad_partials, d.n_partials_node = L.ptr(g_out), L.ptr(g_x1), L.ptr(part), n_pn
    L.call("grl_fbconv_node_bwd", C.byref(d))
    return out, g_x1, part


NODE_SLICES = [("w1", 256 * 64, (256, 64)), ("b1", 256, (256,)), ("w2", 64 * 256, (64, 256)), ("b2", 64, (64,)),
               ("ln_g", 64, (64,)), ("ln_b", 64, (64,)), ("bias", 64, (64,)), ("fk", 16 * 16 * 64, (16, 16, 64))]


def _unpack_node(part):
    g, o, res = part.double().sum(0), 0, {}
    for k, n, shape in NODE_SLICES:
        res[k] = g[o:o + n].view(shape)
        o += n
    return res


def _node_ref(x1, x_dst, p, g_out):
    return R32.node_reference(x1.to(D), x_dst, {k: v.to(D) for k, v in p.items()},
                              grad_out=None if g_out is None else g_out.to(D))


def _node_perturbation_caught(x1, x_dst, p, ref, g_out, tol_out, tol_gx1):
    """The node kernels see no edges, so the stand-in for a lost message is one node losing half of its input: half of
    one orientation row of x1 (what dropping one of two in-edges does to it) must move `out` by >= 5x the tolerance, and
    half of the node's upstream gradient must move its grad_x1 row by >= 5x."""
    k = x1.shape[0] // 2
    x1p = x1.clone()
    x1p[k, 5] *= 0.5
    r = R.row_rel(_node_ref(x1p, x_dst, p, None)["out"] - x_dst.to(D), ref["out"] - x_dst.to(D))
    assert r >= 5 * tol_out, f"half a message moves out by {r:.3e} only"
    if g_out is not None:
        gp = g_out.clone()
        gp[k] *= 0.5
        r = R.row_rel(_node_ref(x1, x_dst, p, gp)["grad"]["x_src"], ref["grad"]["x_src"])
        assert r >= 5 * tol_gx1, f"half a node's upstream gradient moves grad_x1 by {r:.3e} only"


def _node_inputs(n, seed=41):
    g = torch.Generator().manual_seed(seed)
    x1 = (torch.randn(n, 16, 64, generator=g) * 2).cuda()
    x_dst = torch.randn(n, 16, 64, generator=g).cuda()
    g_out = torch.randn(n, 16, 64, generator=g).cuda()
    return x1, x_dst, g_out


def _check_node(tag, x1, x_dst, p, g_out, tol_out=TOL_OUT, tol_gx1=TOL_GX1, counts=None):
    n = x1.shape[0]
    n_tiles = (n + 7) // 8
    ref = _node_ref(x1, x_dst, p, g_out)
    bad, report, first, worst = [], [], None, 0.0
    for n_pn in sorted(counts or {1, 5, n_tiles, n_tiles + 3}):
        out, g_x1, part = _node_launch(x1, x_dst, p, g_out, n_pn)
        again = _node_launch(x1, x_dst, p, g_out, n_pn)
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip((out, g_x1, part), again)), "two identical launches differ"
        got = _unpack_node(part)
        if first is None:
            first = (out, g_x1, got)
            _row(bad, report, "out - x_dst", out - x_dst, ref["out"] - x_dst.to(D), tol_out)
            _row(bad, report, "grad_x1", g_x1, ref["grad"]["x_src"], tol_gx1)
            for k, _, _ in NODE_SLICES:
                _glob(bad, report, f"grad {k}", got[k], ref["grad"][k])
        else:
            assert torch.equal(out, first[0]), f"out depends on n_partials_node={n_pn}"
            assert torch.equal(g_x1, first[1]), f"grad_x1 depends on n_partials_node={n_pn}"
            for k, _, _ in NODE_SLICES:
                worst = max(worst, R.global_rel(got[k], first[2][k]))
                _glob(bad, [], f"n_p={n_pn} grad {k}", got[k], ref["grad"][k], REASSOC)
        if n_pn > n_tiles:
            assert torch.equal(part[n_tiles:], torch.zeros_like(part[n_tiles:])), f"n_p={n_pn}: an idle slot is not 0"
    report.append(f"partial counts: reassociation {worst:.3e} (tol {REASSOC:.0e})")
    if not worst < REASSOC:
        bad.append(f"partial counts move the node gradients by {worst:.3e}")
    _finish(tag, bad, report)
    return ref


def _node_sizes():
    g = 16 * _sms()
    return {"1": 1, "7": 7, "8": 8, "9": 9, "16": 16, "17": 17, "16G-8": g - 8, "16G+8": g + 8, "20011": 20011}


@pytest.mark.parametrize("size", ["1", "7", "8", "9", "16", "17", "16G-8", "16G+8", "20011"])
def test_node_kernels_alone_against_fp64(size):
    n = _node_sizes()[size]
    x1, x_dst, g_out = _node_inputs(n)
    p = _params(8)
    ref = _check_node(f"node n_dst={n}", x1, x_dst, p, g_out)
    _node_perturbation_caught(x1, x_dst, p, ref, g_out, TOL_OUT, TOL_GX1)


@pytest.mark.parametrize("case", ["constant_rows", "offset", "x1*1e-3", "x1*1e3"])
def test_node_kernels_layernorm_rows(case):
    """LayerNorm rows the model produces.  constant_rows: nodes without in-edges at initialisation (x1 = 0, bias = 0)
    give an exactly constant x2 row of variance 0.  offset: bias 30 on every channel over a spread of ~0.2, where a
    one-pass variance would cancel catastrophically; the fp32 value of x2 itself then carries offset/spread * 2^-24.
    x1 at 1e-3 and 1e3 of its scale: the first, uncalibrated forward."""
    n = 1001
    x1, x_dst, g_out = _node_inputs(n, 43)
    p = _params(9)
    tol_out, tol_gx1 = TOL_OUT, TOL_GX1
    if case == "constant_rows":
        p["bias"] = torch.zeros_like(p["bias"])
        x1[::3] = 0
    elif case == "offset":
        p["bias"] = p["bias"] + 30.0
        x2 = torch.einsum("boc,opc->bpc", x1.double(), p["fk"].double()) / 16 + p["bias"].double()
        ratio = float((x2.mean(-1).abs() / x2.std(-1)).max())
        tol_out, tol_gx1 = TOL_OUT + ratio * OFFSET_ULPS * U, TOL_GX1 + ratio * OFFSET_ULPS * U
        print(f"[node offset] offset / spread up to {ratio:.1f}: bounds {tol_out:.2e}, {tol_gx1:.2e}")
    else:
        x1 = x1 * (1e-3 if case == "x1*1e-3" else 1e3)
    ref = _check_node(f"node LayerNorm {case}", x1, x_dst, p, g_out, tol_out, tol_gx1, counts={1, 37})
    if case == "constant_rows":  # x2 = 0 exactly: y = ln_b and the MLP output is the same for every such row
        out, _, _ = _node_launch(x1, torch.zeros_like(x_dst), p, None, 1)
        mlp = out[::3].reshape(-1, 64)
        assert torch.equal(mlp, mlp[0:1].expand_as(mlp)), "constant rows give different outputs"
    _node_perturbation_caught(x1, x_dst, p, ref, g_out, tol_out, tol_gx1)


def test_node_forward_accumulate_out():
    """accumulate_out = 1: out = (x_dst + mlp) + previous out, one fp32 add after the plain store's value."""
    n = 2377
    x1, x_dst, _ = _node_inputs(n, 47)
    p = _params(10)
    prev = torch.randn(n, 16, 64, generator=torch.Generator().manual_seed(2)).cuda()
    out, _, _ = _node_launch(x1, x_dst, p, None, 1)
    out_acc, _, _ = _node_launch(x1, x_dst, p, None, 1, accumulate=prev)
    assert torch.equal(out_acc, out + prev), "accumulate_out is not out = (x_dst + mlp) + previous"
    ref = _node_ref(x1, x_dst, p, None)
    bad, report = [], []
    _row(bad, report, "out - x_dst", out - x_dst, ref["out"] - x_dst.to(D), TOL_OUT)
    _finish("node accumulate", bad, report)


# ---------------------------------------------------------------------------------------------------------------------
# d. the whole strict layer
# ---------------------------------------------------------------------------------------------------------------------
LAYER_GRADS = ["x_src", "x_dst", "bw1", "bb1", "bw2", "bb2", "fk", "wk", "bias", "ln_g", "ln_b", "w1", "b1", "w2", "b2"]


def _strict_layer(es, x_src, x_dst, pos_src, pos_dst, p, dim, w, sub=None):
    """ops.fiber_conv on the fp32 basis of EdgeBasisFn (strict path): (out, {name: grad})."""
    from geometry_rl_b200 import ops
    assert ops.get_precision() == "fp32"
    leaves = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    xs = x_src.clone().requires_grad_(True)
    xd = None if x_dst is None else x_dst.clone().requires_grad_(True)
    basis = ops.EdgeBasisFn.apply(pos_src, pos_dst, leaves["bw1"], leaves["bb1"], leaves["bw2"], leaves["bb2"], _ori(dim),
                                  dim, es)
    assert basis.dtype == torch.float32
    out = ops.fiber_conv(xs, xd, basis, leaves["fk"], leaves["wk"], leaves["bias"], leaves["ln_g"], leaves["ln_b"],
                         leaves["w1"], leaves["b1"], leaves["w2"], leaves["b2"], es, sub)
    out.backward(w)
    grads = {k: v.grad for k, v in leaves.items()}
    grads["x_src"] = xs.grad
    if xd is not None:
        grads["x_dst"] = xd.grad
    return out.detach(), grads


def _compare_layer(tag, es, x_src, x_dst, pos_src, pos_dst, p, dim, w, sub=None):
    out, grads = _strict_layer(es, x_src, x_dst, pos_src, pos_dst, p, dim, w, sub)
    torch.cuda.synchronize()
    ei = torch.stack([es.edge_src.long(), es.edge_dst.long()])
    kw = dict(x_src=x_src.to(D), x_dst=None if x_dst is None else x_dst.to(D), pos_src=pos_src.to(D),
              pos_dst=pos_dst.to(D), params={k: v.to(D) for k, v in p.items()}, ori3=_ori(dim).to(D), dim=dim,
              out_ids=None if sub is None else sub.out_ids)
    ref = R.layer_reference(edge_index=ei, grad_out=w.to(D), **kw)
    resid = (x_src if sub is None else x_src[sub.out_ids]) if x_dst is None else x_dst
    bad, report = [], [f"{es.n_src} src, {es.n_dst} dst, {es.n_edges} edges"]
    _glob(bad, report, "out", out, ref["out"], NORTH_STAR)
    r_out = _row(bad, report, "out - x_dst", out - resid, ref["out"] - resid.to(D), TOL_OUT)
    for k in LAYER_GRADS:
        if k == "x_dst" and x_dst is None:
            continue
        _glob(bad, report, f"grad {k}", grads[k], ref["grad"][k], NORTH_STAR)
    _finish(f"layer {tag}", bad, report)
    if sub is not None:  # perturb one of the edges the sub layer reads
        ei = ei[:, torch.isin(ei[1], sub.out_ids)]
    for kind, res in R.perturbed(R.layer_reference, ei, x_src.shape[0], **kw).items():
        r = R.row_rel(res["out"] - resid.to(D), ref["out"] - resid.to(D))
        assert r >= 5 * TOL_OUT, f"{tag}: one {kind} edge moves out by only {r:.3e} < 5 x {TOL_OUT:g}"
    return r_out


def _random_edge_set(B, ns, nd, e_per, seed, homo):
    from geometry_rl_b200 import ops
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(0, ns, (B, e_per), generator=g)
    dst = torch.randint(0, nd, (B, e_per), generator=g)
    if homo:
        src, dst = src.clamp_max(ns - 2), dst.clamp_max(nd - 2)  # a few nodes without edges
    coo = torch.stack([(src + (torch.arange(B) * ns)[:, None]).reshape(-1), (dst + (torch.arange(B) * nd)[:, None]).reshape(-1)])
    coo = coo[:, torch.sort(coo[0] * (B * nd) + coo[1]).indices]
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
def test_strict_layer_against_fp64(kind):
    from geometry_rl_b200 import ops
    if kind == "bipartite":
        es = _random_edge_set(16, 30, 7, 90, 61, False)
        x_src, x_dst, pos_src, pos_dst, w = _layer_inputs(es.n_src, es.n_dst, es.n_dst, 62)
        _compare_layer(kind, es, x_src, x_dst, pos_src, pos_dst, _params(12), 3, w)
        return
    es = _random_edge_set(40, 49, 49, 128, 63, True)
    sub = ops.build_sub_edge_set(es, (torch.arange(40) * 49 + 3).cuda()) if kind == "sub" else None
    x_src, _, pos_src, _, w = _layer_inputs(es.n_src, 1, es.n_dst if sub is None else sub.n_dst, 64)
    _compare_layer(kind, es, x_src, None, pos_src, pos_src, _params(13), 2, w, sub)


def _two_layer_reference(x, pos, p1, p2, dim, ei, w):
    """Two homogeneous layers on ONE basis (the basis MLP of p1), fp64 autograd: out and grad[name] of x, the basis MLP
    (summed over both layers by autograd) and the layer parameters as "1.<name>" / "2.<name>"."""
    from oracle import models as om
    leaves = {"x": x.to(D).requires_grad_(True)}
    for i, p in ((1, p1), (2, p2)):
        for k, v in p.items():
            if k not in R32.BASIS or i == 1:
                leaves[k if k in R32.BASIS else f"{i}.{k}"] = v.to(D).requires_grad_(True)
    sp, _ = om.invariants(_ori(dim)[:, :dim].to(D), pos[ei[0]][:, :dim].to(D), pos[ei[1]][:, :dim].to(D))
    kb = om.basis_mlp(sp, {"basis_fn.1.weight": leaves["bw1"], "basis_fn.1.bias": leaves["bb1"],
                           "basis_fn.3.weight": leaves["bw2"], "basis_fn.3.bias": leaves["bb2"]}, "basis_fn")
    h = leaves["x"]
    eye = torch.eye(64, dtype=D, device="cuda")
    for i in (1, 2):
        q = {k: leaves[f"{i}.{k}"] for k in R.PARAM_NAMES if k not in R32.BASIS}
        sd = {"c.kernel.weight": q["wk"], "c.fiber_kernel.weight": eye, "c.bias": q["bias"], "c.m.0.weight": q["ln_g"],
              "c.m.0.bias": q["ln_b"], "c.m.1.weight": q["w1"], "c.m.1.bias": q["b1"], "c.m.3.weight": q["w2"],
              "c.m.3.bias": q["b2"]}
        x2 = om.fiber_bundle_conv(h, h, ei, kb, q["fk"], sd, "c")
        h = om.convnext_update(h, x2, sd, "c.m.0", "c.m.1", "c.m.3")
    names = list(leaves)
    gs = torch.autograd.grad(h, [leaves[k] for k in names], w.to(D))
    return h.detach(), dict(zip(names, gs))


def test_strict_layer_two_layers_sharing_one_basis():
    """Two layers on one EdgeBasisFn output: autograd sums the two [E,16,64] basis gradients before grl_edge_basis_bwd."""
    from geometry_rl_b200 import ops
    es = _random_edge_set(24, 33, 33, 96, 65, True)
    x, _, pos, _, w = _layer_inputs(es.n_src, 1, es.n_dst, 66)
    p1, p2 = _params(18), _params(19)
    leaves = {"x": x.clone().requires_grad_(True)}
    for k in R.PARAM_NAMES:
        if k in R32.BASIS:
            leaves[k] = p1[k].clone().requires_grad_(True)
        else:
            leaves[f"1.{k}"], leaves[f"2.{k}"] = p1[k].clone().requires_grad_(True), p2[k].clone().requires_grad_(True)
    basis = ops.EdgeBasisFn.apply(pos, pos, leaves["bw1"], leaves["bb1"], leaves["bw2"], leaves["bb2"], _ori(3), 3, es)
    h = leaves["x"]
    for i in (1, 2):
        q = {k: leaves[f"{i}.{k}"] for k in R.PARAM_NAMES if k not in R32.BASIS}
        h = ops.fiber_conv(h, None, basis, q["fk"], q["wk"], q["bias"], q["ln_g"], q["ln_b"], q["w1"], q["b1"], q["w2"],
                           q["b2"], es)
    h.backward(w)
    ei = torch.stack([es.edge_src.long(), es.edge_dst.long()])
    ref_out, ref_g = _two_layer_reference(x, pos, p1, p2, 3, ei, w)
    bad, report = [], []
    _glob(bad, report, "out", h, ref_out, NORTH_STAR)
    for k, v in leaves.items():
        _glob(bad, report, f"grad {k}", v.grad, ref_g[k], NORTH_STAR)
    _finish("layer two layers, one basis", bad, report)


def _builder_graph(name, B, seed):
    from geometry_rl_b200.synthetic import CONFIGS, synthetic_obs
    cfg = CONFIGS[name]
    obs = synthetic_obs(cfg, B, torch.Generator().manual_seed(seed), env_ids=torch.arange(B) % cfg.num_envs)
    graph, _ = G.make_data(cfg, policy=True).build_data(*G.obs_args(cfg, obs, policy=True), train=False)
    return cfg, graph


@pytest.mark.parametrize("et", ["internal", "task"])
def test_strict_layer_hepi_topology(et):
    """The HEPi builder's rigid-insertion edge types at minibatch 256: internal (homogeneous) and TASK (bipartite)."""
    from geometry_rl_b200 import ops
    cfg, graph = _builder_graph("rigid_insertion_multi_hepi_trpl_cfg", 256, 25)
    key = ("object_geometry", "internal", "object_geometry") if et == "internal" else \
        ("object_geometry", "task", "grippers")
    es = ops.exact_edge_set(graph.edge_sets[key])
    pos_src, pos_dst = graph[key[0]].pos.float().contiguous(), graph[key[2]].pos.float().contiguous()
    x_src, x_dst, _, _, w = _layer_inputs(es.n_src, es.n_dst, es.n_dst, 67)
    _compare_layer(f"hepi {et}", es, x_src, None if et == "internal" else x_dst, pos_src,
                   pos_src if et == "internal" else pos_dst, _params(21), cfg.ponita_dim, w)


@pytest.mark.parametrize("kind", ["dense", "pruned_sub"])
def test_strict_layer_empn_topology(kind):
    """The EMPN builder's homogeneous view (rigid pushing, minibatch 128), and its pruned set with the last layer's
    sub set (edges into the output nodes only)."""
    from geometry_rl_b200 import ops
    cfg, graph = _builder_graph("rigid_pushing_multi_empn_trpl_cfg", 128, 27)
    B = len(graph)
    pos = torch.cat([graph[t].pos.reshape(B, -1, 3) for t in graph.node_types], dim=1).reshape(-1, 3).float()
    if kind == "dense":
        es, sub = ops.exact_edge_set(graph.homogeneous()), None
    else:
        pr = graph.homogeneous_pruned()
        es = ops.exact_edge_set(pr.es)
        sub = pr.sub if pr.sub.exact else ops.build_sub_edge_set(es, pr.sub.out_ids)
        if pr.live_ids is not None:
            pos = pos[pr.live_ids]
    pos = pos.contiguous()
    x_src, _, _, _, w = _layer_inputs(es.n_src, 1, es.n_dst if sub is None else sub.n_dst, 68)
    _compare_layer(f"empn {kind}", es, x_src, None, pos, pos, _params(22), cfg.ponita_dim, w, sub)


# ---------------------------------------------------------------------------------------------------------------------
# e. the one-time calibration
# ---------------------------------------------------------------------------------------------------------------------
def _calib_case(seed, homo=True):
    es = _random_edge_set(32, 41, 41 if homo else 9, 120, seed, homo)
    x_src, x_dst, pos_src, pos_dst, _ = _layer_inputs(es.n_src, es.n_dst, 1, seed + 1)
    return es, x_src, (None if homo else x_dst * 1.7), pos_src, (pos_src if homo else pos_dst)


def _precision(mode):
    from geometry_rl_b200 import ops

    class _P:
        def __enter__(self):
            ops.set_precision(mode)

        def __exit__(self, *a):
            ops.set_precision("fp32")
    return _P()


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_aggregate_messages_against_fp64(mode):
    """ops.aggregate_messages on a BasisSpec alone: fp32 mode materialises the basis with grl_edge_basis_fwd, bf16 mode
    with grl_edge_basis_fwd_tc (bf16), converted to fp32 and fed to grl_fbconv_edge_fwd in both."""
    from geometry_rl_b200 import ops
    es, x_src, _, pos_src, pos_dst = _calib_case(71, homo=False)
    p = _params(23)
    dim = 3
    ei = torch.stack([es.edge_src.long(), es.edge_dst.long()])
    with _precision(mode):
        spec = ops.BasisSpec(pos_src, pos_dst, p["bw1"], p["bb1"], p["bw2"], p["bb2"], _ori(dim), dim, es)
        basis = spec.materialize()
        x1 = ops.aggregate_messages(x_src, spec, p["wk"], es)
    torch.cuda.synchronize()
    assert basis.dtype == (torch.bfloat16 if mode == "bf16" else torch.float32)
    kw = dict(pos_src=pos_src.to(D), pos_dst=pos_dst.to(D), params=p, ori3=_ori(dim).to(D), dim=dim)
    ref_b = R32.basis_reference(edge_index=ei, **kw)["basis"]
    ref = R.edge_reference(x_src=x_src.to(D), n_dst=es.n_dst, edge_index=ei, **kw)["x1"]
    deg = int((es.rowptr_dst[1:] - es.rowptr_dst[:-1]).max())
    tol_b, tol_x1 = (TOL_BASIS16, TOL_X1_16) if mode == "bf16" else (TOL_BASIS, _deg_tol(TOL_X1, deg))
    bad, report = [], []
    _row(bad, report, "basis", basis, ref_b, tol_b)
    _row(bad, report, "x1", x1, ref, tol_x1)
    _finish(f"aggregate_messages {mode}", bad, report)
    for kind, pe in R.perturbed(R.edge_reference, ei, es.n_src, x_src=x_src.to(D), n_dst=es.n_dst, **kw).items():
        assert R.row_rel(pe["x1"], ref) >= 5 * tol_x1, f"one {kind} edge not caught"


def _hepi_conv(seed):
    from geometry_rl_b200.modules.pyg_models.ponita.conv import FiberBundleConv
    torch.manual_seed(seed)
    return FiberBundleConv(64, 64, 64, groups=64, separable=True, widening_factor=4).cuda()


def _empn_layer(seed):
    from geometry_rl_b200.modules.pyg_models.ponita.ponita import SeparableFiberBundleConvNext
    torch.manual_seed(seed)
    return SeparableFiberBundleConvNext(64, 64, layer_scale=None).cuda()


def _basis_mlp(seed):
    p = _params(seed)
    return {k: torch.nn.Parameter(p[k]) for k in R32.BASIS}


def _factors_reference(x_src, x_dst, pos_src, pos_dst, bp, wk, fk_op, dim, es):
    ei = torch.stack([es.edge_src.long(), es.edge_dst.long()])
    params = dict({k: v.detach() for k, v in bp.items()}, wk=wk.detach())
    x1 = R.edge_reference(x_src=x_src.to(D), pos_src=pos_src.to(D), pos_dst=pos_dst.to(D), params=params,
                          ori3=_ori(dim).to(D), dim=dim, edge_index=ei, n_dst=es.n_dst)["x1"]
    return R32.calibration_reference(x_dst.to(D), x1, fk_op.detach().to(D))


# relative error of the factors: fp32 measured 1.0e-7; the bf16 basis (relative step 2^-8, tanh GELU) moves them by up
# to 1.9e-4 (EMPN std_in/std_1), 1.4e-4 on the capacity radius set
TOL_FACTOR = {"fp32": 1e-6, "bf16": 1e-3}


@pytest.mark.parametrize("model", ["hepi", "empn"])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_calibration_factors_and_module_behaviour(model, mode):
    """The factors against fp64; then the first training forward runs on the un-calibrated weights (bit-identical to
    ops.fiber_conv with them), rescales kernel.weight and fiber_kernel.weight by exactly the factors and sets
    `callibrated`; the second forward runs on the scaled weights."""
    from geometry_rl_b200 import ops
    homo = model == "empn"
    es, x_src, x_dst, pos_src, pos_dst = _calib_case(73 if homo else 75, homo)
    dim = 3
    bp = _basis_mlp(24)
    fb = (torch.rand(16, 16, 64, generator=torch.Generator().manual_seed(5)) * 0.5).cuda()  # a fibre basis
    with _precision(mode):
        basis = ops.edge_basis(pos_src, pos_dst, bp["bw1"], bp["bb1"], bp["bw2"], bp["bb2"], _ori(dim), dim, es)
        if model == "hepi":
            mod = _hepi_conv(31).train()
            c, fk_of = mod, lambda: F.linear(fb, mod.fiber_kernel.weight)
            run = lambda: mod((x_src, x_dst), edge_attr=basis, fiber_attr=fb, edge_set=es)[1]  # noqa: E731
        else:
            mod = _empn_layer(32).train()
            c, fk_of = mod.conv, lambda: F.linear(fb, mod.conv.fiber_kernel.weight).transpose(0, 1).contiguous()
            run = lambda: mod(x_src, basis, fb, es)  # noqa: E731
        w0, f0 = c.kernel.weight.detach().clone(), c.fiber_kernel.weight.detach().clone()
        xd = x_src if x_dst is None else x_dst
        if model == "hepi":
            fac = mod._callibration_factors(x_src, xd, basis, fk_of(), es)
        else:
            fac = mod._callibration_factors(x_src, basis, fk_of(), es)
        ref = _factors_reference(x_src, xd, pos_src, pos_dst, bp, w0, fk_of(), dim, es)
        errs = [abs(float(a) / float(b) - 1) for a, b in zip(fac, ref)]
        print(f"[calibration {model} {mode}] std_in/std_1 {float(fac[0]):.6f} vs fp64 {float(ref[0]):.6f} (rel "
              f"{errs[0]:.2e}); std_1/std_2 {float(fac[1]):.6f} vs {float(ref[1]):.6f} (rel {errs[1]:.2e}); "
              f"tol {TOL_FACTOR[mode]:.0e}")
        assert max(errs) < TOL_FACTOR[mode], errs

        def plain(wk, fw):
            fk = F.linear(fb, fw)
            if model == "empn":
                fk = fk.transpose(0, 1).contiguous()
                lin = (mod.norm.weight, mod.norm.bias, mod.linear_1.weight, mod.linear_1.bias, mod.linear_2.weight,
                       mod.linear_2.bias)
            else:
                m = mod.node_mlp
                lin = (m[0].weight, m[0].bias, m[1].weight, m[1].bias, m[3].weight, m[3].bias)
            return ops.fiber_conv(x_src, x_dst, basis, fk, wk, c.bias, *lin, es)

        with torch.no_grad():
            out1 = run()
            assert bool(c.callibrated), "the first training forward did not set callibrated"
            assert torch.equal(out1, plain(w0, f0)), "the first forward did not use the un-calibrated weights"
            assert torch.equal(c.kernel.weight, w0 * fac[0]) and torch.equal(c.fiber_kernel.weight, f0 * fac[1]), \
                "the weights are not rescaled by the factors"
            out2 = run()
            assert torch.equal(out2, plain(w0 * fac[0], f0 * fac[1])), "the second forward does not use the scaled weights"


def test_calibration_on_a_capacity_radius_set():
    """bf16: the factors of a fixed-capacity radius set equal those of the exact set built from the same edges; a
    capacity set with no real edge returns None and leaves `callibrated` False through a training forward."""
    from geometry_rl_b200 import ops
    B, P, r, m = 12, 40, 0.45, 6
    g = torch.Generator().manual_seed(77)
    pos = (torch.randn(B, P, 3, generator=g) * 0.5).cuda()
    pos_f = pos.reshape(-1, 3).contiguous()
    x = torch.randn(B * P, 16, 64, generator=g).cuda()
    bp = _basis_mlp(25)
    fb = (torch.rand(16, 16, 64, generator=g) * 0.5).cuda()
    conv = _hepi_conv(33).train()
    fk = F.linear(fb, conv.fiber_kernel.weight)
    with _precision("bf16"), torch.no_grad():
        nv = torch.tensor([40, 0, 33, 40, 17, 40, 40, 2, 40, 40, 39, 40], dtype=torch.int32).cuda()
        coo, ptr = ops.radius_graph(pos, nv, r, m, capacity=B * P * m)
        E = int(ptr[-1])
        es_cap = ops.build_edge_set(coo, ptr, B, P, P, exact=False)
        es_ex = ops.build_edge_set(coo[:, :E].contiguous(), ptr, B, P, P)
        spec = lambda es: ops.BasisSpec(pos_f, pos_f, bp["bw1"], bp["bb1"], bp["bw2"], bp["bb2"], _ori(3), 3, es)  # noqa
        f_cap = conv._callibration_factors(x, x, spec(es_cap), fk, es_cap)
        f_ex = conv._callibration_factors(x, x, spec(es_ex), fk, es_ex)
        assert torch.equal(f_cap[0], f_ex[0]) and torch.equal(f_cap[1], f_ex[1]), (f_cap, f_ex)
        ref = _factors_reference(x, x, pos_f, pos_f, bp, conv.kernel.weight, fk, 3, es_ex)
        errs = [abs(float(a) / float(b) - 1) for a, b in zip(f_cap, ref)]
        print(f"[calibration capacity radius bf16] factors rel to fp64 {errs[0]:.2e}, {errs[1]:.2e}")
        assert max(errs) < TOL_FACTOR["bf16"], errs
        # no real edge at all
        nv0 = torch.zeros(B, dtype=torch.int32, device="cuda")
        coo0, ptr0 = ops.radius_graph(pos, nv0, r, m, capacity=B * P * m)
        es0 = ops.build_edge_set(coo0, ptr0, B, P, P, exact=False)
        assert int(ptr0[-1]) == 0
        assert conv._callibration_factors(x, x, spec(es0), fk, es0) is None
        w0 = conv.kernel.weight.detach().clone()
        conv(x, edge_attr=spec(es0), fiber_attr=fb, edge_set=es0)
        assert not bool(conv.callibrated) and torch.equal(conv.kernel.weight, w0), "an edgeless batch calibrated the conv"
