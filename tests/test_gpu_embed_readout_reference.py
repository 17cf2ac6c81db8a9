"""GPU: the embedding and readout kernels alone against fp64 references (tests/embed_readout_reference.py), with a
per-row metric, at tile, grid-stride and partial edges and on the live-row path.

a. grl_embed_fwd / _bwd through the C ABI, operands packed as ops.EmbedFn packs them: x row by row and the weight
   gradient; F = S + V over every FQ instantiation and its edges (S = 0, V = 0, the data builders' splits), both dims
   (vectors carry a z that must not reach x in 2-D), N around the 16-node tile and the forward's 8 x SMs (FQ <= 2) and
   6 x SMs (FQ >= 3) grid strides; features at 1e-3, 1e3 and mixed column scales; zero feature rows; partial counts 1,
   3, EmbedFn's and n_tiles + 5; the node_ids path on repeated, out-of-order ids into NaN-padded arrays and on the
   rope builder's live rows, bit for bit against the dense launch on the gathered rows.
b. grl_readout_fwd / _bwd through the C ABI, operands packed as ops.ReadoutFn packs them: out and hidden per node,
   grad_latent per (node, orientation) row, decoder gradients; (od, odv) at the gate's two forms up to od + odv = 8,
   both dims, n around the 8-node block and the forward's 4 x SMs grid stride; grad_hidden null and set; a z in
   grad_out that must reach nothing in 2-D; latents with a large common offset and at 1e-3 / 1e3; partial counts 1,
   ReadoutFn's and past ceil(n / 8); the torch formulation taking over, without a launch, where the kernel refuses.

Every output and partial buffer is filled with NaN before a launch; grids and N are sized from _lib.sm_count() at run
time.  Exact properties (zero rows, z = 0, idle slots, repeatability, bit-identity across partial counts and between
the live-row and dense launches) use torch.equal.  Every per-row bound is shown to put a single-row perturbation (one
node's feature dropped, one node's orientation rows swapped or dropped) at 5x or more of it.

Error model and tolerances (u = 2^-24).  The 3-D grid is the upper hemisphere of the rigid insertion config, whose
mean orientation (z 0.5) makes the bias term b_j * mean_o ori[o] of the vector readout visible.
- x: one lifted feature is <v, o> in at most 3 fp32 products (2u |v| |o| absolute), then an F-term FFMA chain per
  channel: (F + 2) u sum_f |feat_f W_cf| per element.  row_rel divides by the row max plus 1% of the tensor's max, so a
  row whose features all nearly vanish at one orientation (a vector nearly orthogonal to it) is held against that floor;
  that row's feature carries its full 2u |v| absolute error: TOL_X = 1e-5 covers both.
- grad_weight of the embedding: each thread sums its CTA's nodes in sequence, then 16 orientations, then the partials
  (summed in fp64 here, by grl_reduce_partials in EmbedFn): held globally (GLOBAL_W) at EmbedFn's count; n_partials = 1
  makes one thread sum all 200003 nodes in sequence, held to REASSOC like every other count.
- hidden: a 16-term sum times 1/16 (exact): 15 u sum_o |l_o| / 16 per element, TOL_HID.
- out: mean_o l ori in a 16-term FMA chain, 64-term dot products reduced over the warp, the bias term, times the gate
  (itself a 64-term dot product): about 25 u of the summed magnitudes; the kernels sum mean_o ori[o], the factor of
  b_j, in double, since the circle's ~1e-8 mean is below the rounding of an fp32 sum.  With od = 1 one gate scales the node's whole
  row, so a node whose gate cancels carries the gate's absolute error, about 8 u sum_c |w_c h_c|, against 1% of the
  largest output: ~200 u, TOL_OUT.  A common offset m over a spread s cancels in sum_o l ori[o] (the circle's means are
  ~0): the partial sums of the FMA chain reach ~3 m, so each of the 64 channels of V carries ~30 m u against a true
  ~2.8 s, and the errors, sharing m and the grid, add up in the 64-term dot product: ~65 (m/s) u, hence the offset
  term (m/s) OFFSET_ULPS u on every per-row bound of that case.
- grad_latent: g_hid + sum_d gV[d] ori[o][d] of short sums (odv + 4 terms); rows where they cancel are held against
  the floor, as for out: TOL_GLAT.
- readout decoder gradients: per-warp sequential sums over the warp's nodes, 8 warps, then the partials: GLOBAL_W.
Worst cases measured on one B200 (1000 W power limit) over every case of this file are recorded next to each bound.
The file runs in about 12 s there."""
import ctypes as C
import math

import pytest
import torch

from tests import conv16_reference as R
from tests import embed_readout_reference as ER
from tests import gpu_helpers as G

pytestmark = pytest.mark.gpu

D = torch.float64
NAN = float("nan")
U = 2.0 ** -24
# per-row (row_rel, floor 1e-2) bounds, measured worst case (case)
TOL_X = 1e-5          # x rows of grl_embed_fwd: 2.8e-6 (N 18943, S 0, V 1, dim 3)
TOL_HID = 4e-6        # hidden rows of grl_readout_fwd: 3.9e-7 (n 16391)
TOL_OUT = 3e-5        # out rows (one node) of grl_readout_fwd: 6.3e-6 (n 2369, od 1, odv 7, dim 3)
TOL_GLAT = 2e-5       # grad_latent rows (one node, one orientation) of grl_readout_bwd: 3.8e-6 (n 4737, od 1, odv 3)
# offset term of the readout, TOL + m/s * OFFSET_ULPS * 2^-24: out 9.1e-5 of 2.0e-4 at m/s = 30 (2-D, od = odv = 1),
# 51 (m/s) u; every other tensor of that case stays below 2.3e-6
OFFSET_ULPS = 96
# global max-norm bound of the weight gradients at the partial counts of EmbedFn / ReadoutFn: 5.6e-7 (embedding,
# N 200003, S 8, V 8), 4.9e-6 (readout bias, n 2369, od 1, odv 3, dim 2)
GLOBAL_W = 5e-5
# any other partial count against fp64, and its distance to the default count: 1.3e-5 (embedding, n_partials = 1 at
# N 200003: one thread sums every node), 5.1e-6 (readout)
REASSOC = 2e-4

_ORI = {}


def _ori(dim):
    """[16,3] orientation grid as ops takes it: the circle in 2-D, the upper hemisphere in 3-D (rigid insertion)."""
    if dim not in _ORI:
        from geometry_rl_b200.modules.pyg_models.ponita.ponita import make_ori_grid, pad_ori3
        _ORI[dim] = pad_ori3(make_ori_grid(dim, 16, dim == 3).cuda()).contiguous()
    return _ORI[dim]


def _sms():
    from geometry_rl_b200 import _lib as L
    return L.sm_count()


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


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
# a. embedding
# ---------------------------------------------------------------------------------------------------------------------
def _embed_desc(n, sc, vc, dim, node_ids=None, **kw):
    from geometry_rl_b200 import _lib as L
    return L.GrlEmbedDesc(n_nodes=n, n_scalars=sc.shape[1], n_vectors=vc.shape[1] // 3, dim=dim, scalars=L.ptr(sc),
                          vectors=L.ptr(vc), ori=L.ptr(_ori(dim)), node_ids=L.ptr(node_ids),
                          **{k: L.ptr(v) if isinstance(v, torch.Tensor) else v for k, v in kw.items()})


def _embed_fwd(sc, vc, w, dim, node_ids=None):
    from geometry_rl_b200 import _lib as L
    n = sc.shape[0] if node_ids is None else node_ids.numel()
    x = torch.full((n, 16, 64), NAN, device="cuda")
    L.call("grl_embed_fwd", C.byref(_embed_desc(n, sc, vc, dim, node_ids, weight=w, x=x)))
    return x


def _embed_bwd(sc, vc, g_x, dim, n_p, node_ids=None):
    """The partial slots [n_p, 64, S+V] of grl_embed_bwd."""
    from geometry_rl_b200 import _lib as L
    n, F = g_x.shape[0], sc.shape[1] + vc.shape[1] // 3
    part = torch.full((n_p, 64, F), NAN, device="cuda")
    L.call("grl_embed_bwd", C.byref(_embed_desc(n, sc, vc, dim, node_ids, grad_x=g_x, grad_weight_partials=part,
                                                n_partials=n_p)))
    return part


def _embed_np(n, F):
    """EmbedFn's partial count (resident CTAs per SM of grl_embed_bwd)."""
    return max(1, min((n + 15) // 16, (4 if F <= 8 else 2) * _sms()))


def _embed_inputs(n, S, V, seed, scale=1.0):
    """Features ~N(0, scale) (a per-column scale vector for "mixed"), z non-zero; every 97th node (from the 41st) has
    all-zero features; weight ~N(0, 1/F) like an initialised Linear; grad_x ~N(0, 1)."""
    g = _gen(seed)
    F = S + V
    cs = torch.as_tensor(scale, dtype=torch.float32, device="cuda").expand(F)
    sc = torch.randn(n, S, generator=g, device="cuda") * cs[:S]
    vc = (torch.randn(n, V, 3, generator=g, device="cuda") * cs[S:, None]).reshape(n, 3 * V)
    zero = torch.arange(n, device="cuda") % 97 == 41
    sc[zero], vc[zero] = 0.0, 0.0
    w = torch.randn(64, F, generator=g, device="cuda") / math.sqrt(F)
    g_x = torch.randn(n, 16, 64, generator=g, device="cuda")
    return sc.contiguous(), vc.contiguous(), w.contiguous(), g_x, zero


def _embed_ref(sc, vc, w, dim, node_ids=None, g_x=None):
    return ER.embed_reference(sc.to(D), vc.to(D), w.to(D), _ori(dim).to(D), dim, node_ids,
                              None if g_x is None else g_x.to(D))


def _dropped_feature(sc, vc, node):
    """Node `node` loses its largest feature (a vector when it has one): the single-row perturbation of the embedding."""
    sc, vc = sc.clone(), vc.clone()
    V = vc.shape[1] // 3
    if V:
        v = int(vc[node].view(V, 3).norm(dim=1).argmax())
        vc[node, 3 * v:3 * v + 3] = 0
    else:
        sc[node, int(sc[node].abs().argmax())] = 0
    return sc, vc


def _check_embed(tag, sc, vc, w, g_x, dim, zero=None, counts=True, perturb=True, node_ids=None):
    n, F = g_x.shape[0], w.shape[1]
    n_tiles = (n + 15) // 16
    n_p0 = _embed_np(n, F)
    x = _embed_fwd(sc, vc, w, dim, node_ids)
    part = _embed_bwd(sc, vc, g_x, dim, n_p0, node_ids)
    torch.cuda.synchronize()
    ref = _embed_ref(sc, vc, w, dim, node_ids, g_x)
    bad, report = [], [f"N={n} S={sc.shape[1]} V={vc.shape[1] // 3} dim={dim}"]
    _row(bad, report, "x", x, ref["x"], TOL_X)
    gw = part.double().sum(0)
    _glob(bad, report, "grad weight", gw, ref["grad_weight"])
    if zero is not None and bool(zero.any()):
        assert torch.equal(x[zero], torch.zeros_like(x[zero])), "x of a node with zero features is not 0"
    # exact: a second launch gives the same bits
    assert torch.equal(x, _embed_fwd(sc, vc, w, dim, node_ids)), "forward not repeatable"
    assert torch.equal(part, _embed_bwd(sc, vc, g_x, dim, n_p0, node_ids)), "backward not repeatable"
    if dim == 2 and vc.shape[1]:  # a different z changes no bit
        vz = vc.clone().view(vc.shape[0], -1, 3)
        vz[..., 2] = vz[..., 2] * -3.0 + 7.0
        vz = vz.view(vc.shape)
        assert torch.equal(x, _embed_fwd(sc, vz, w, dim, node_ids)), "the z of a vector reaches x in 2-D"
        assert torch.equal(part, _embed_bwd(sc, vz, g_x, dim, n_p0, node_ids)), "the z of a vector reaches grad W in 2-D"
    worst = 0.0
    for n_p in sorted({1, 3, n_tiles + 5} if counts else set()):
        pp = _embed_bwd(sc, vc, g_x, dim, n_p, node_ids)
        gp = pp.double().sum(0)
        worst = max(worst, R.global_rel(gp, gw))
        _glob(bad, [], f"n_partials={n_p} grad weight", gp, ref["grad_weight"], REASSOC)
        if n_p > n_tiles:
            assert torch.equal(pp[n_tiles:], torch.zeros_like(pp[n_tiles:])), f"n_partials={n_p}: idle slot not 0"
    if counts:
        report.append(f"partial counts: reassociation {worst:.3e} (tol {REASSOC:.0e})")
        if not worst < REASSOC:
            bad.append(f"partial counts move grad weight by {worst:.3e}")
    _finish(tag, bad, report)
    if perturb:  # the per-row bound catches one node (the last, in the last, possibly partial tile) losing a feature
        k = n - 1 if node_ids is None else int(node_ids[-1])
        if zero is not None and bool(zero[k]):
            return ref
        r = R.row_rel(_embed_ref(*_dropped_feature(sc, vc, k), w, dim, node_ids)["x"], ref["x"])
        assert r >= 5 * TOL_X, f"{tag}: one dropped feature moves x by {r:.3e} only"
    return ref


# (S, V): every FQ = ceil(F / 4) and its edges, S = 0 and V = 0, and the data builders' splits (rigid 3 + 4, cloth
# 4 + 3, rope 3 + 3; test_embed_builders_features checks that list against the builders)
EMBED_SPLITS = [(0, 1), (1, 0), (4, 0), (2, 3), (3, 3), (3, 4), (4, 3), (4, 4), (5, 4), (6, 6), (0, 13), (8, 8)]


def _embed_sizes():
    s = _sms()
    return [1, 15, 16, 17, 8 * s * 16 - 1, 8 * s * 16 + 1, 6 * s * 16 + 1, 200003]


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("S,V", EMBED_SPLITS, ids=[f"S{s}V{v}" for s, v in EMBED_SPLITS])
def test_embed_kernels_alone_against_fp64(S, V, dim):
    for n in _embed_sizes():
        sc, vc, w, g_x, zero = _embed_inputs(n, S, V, 1000 * S + 10 * V + dim + n)
        _check_embed(f"embed N={n} S={S} V={V} dim={dim}", sc, vc, w, g_x, dim, zero)


@pytest.mark.parametrize("scale", ["1e-3", "1e3", "mixed"])
@pytest.mark.parametrize("S,V", [(3, 4), (8, 8)])
def test_embed_feature_scales(S, V, scale):
    """Features at 1e-3 and 1e3 of unit scale, and columns alternating between the two (one row then spans 1e6)."""
    n = 8 * _sms() * 16 + 1
    cs = {"1e-3": 1e-3, "1e3": 1e3}.get(scale) or [1e-3 if f % 2 else 1e3 for f in range(S + V)]
    for dim in (2, 3):
        sc, vc, w, g_x, zero = _embed_inputs(n, S, V, 77 + dim, cs)
        _check_embed(f"embed scale {scale} S={S} V={V} dim={dim}", sc, vc, w, g_x, dim, zero, counts=False)


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("S,V", [(0, 5), (3, 4), (8, 8)])
def test_embed_live_rows(S, V, dim):
    """node_ids that repeat and run out of order into padded arrays whose other rows are NaN: x and every partial slot
    bit-identical to the dense launch on the gathered rows, at EmbedFn's count and at 3; fp64 on the live rows."""
    n_pad, n = 9001, 7001
    g = _gen(5 + S + V + dim)
    sc, vc, w, _, _ = _embed_inputs(n_pad, S, V, 9 + dim)
    dead = torch.arange(n_pad, device="cuda") % 7 == 3
    alive = (~dead).nonzero().squeeze(1)
    ids = alive[torch.randint(0, alive.numel(), (n,), generator=g, device="cuda")]
    ids[:40] = ids[:40].flip(0)
    ids[100:140] = alive[5]  # one row read 40 times
    ids = ids.int().contiguous()
    sc[dead], vc[dead] = NAN, NAN
    g_x = torch.randn(n, 16, 64, generator=g, device="cuda")
    _check_embed(f"embed live rows S={S} V={V} dim={dim}", sc, vc, w, g_x, dim, node_ids=ids, counts=False)
    _same_as_dense(sc, vc, w, g_x, dim, ids)


def _same_as_dense(sc, vc, w, g_x, dim, ids):
    n = ids.numel()
    scg, vcg = sc[ids.long()].contiguous(), vc[ids.long()].contiguous()
    assert torch.equal(_embed_fwd(sc, vc, w, dim, ids), _embed_fwd(scg, vcg, w, dim)), "live-row x differs from dense"
    for n_p in (_embed_np(n, w.shape[1]), 3):
        assert torch.equal(_embed_bwd(sc, vc, g_x, dim, n_p, ids), _embed_bwd(scg, vcg, g_x, dim, n_p)), \
            f"live-row grad W partials differ from dense at n_partials={n_p}"


def _builder_features(name, B=64):
    from geometry_rl_b200.synthetic import CONFIGS, synthetic_obs
    cfg = CONFIGS[name]
    obs = synthetic_obs(cfg, B, torch.Generator().manual_seed(21), env_ids=torch.arange(B) % cfg.num_envs)
    graph, u = G.make_data(cfg, policy=True).build_data(*G.obs_args(cfg, obs, policy=True), train=False)
    return cfg, graph, u


BUILDERS = ["rigid_insertion_multi_hepi_trpl_cfg", "rigid_pushing_multi_empn_trpl_cfg",
            "cloth_hanging_multi_hepi_trpl_cfg", "rope_shaping_hepi_trpl_cfg"]


@pytest.mark.parametrize("name", BUILDERS)
def test_embed_builders_features(name):
    """The features the data builders produce, at the config's dim, with the (S, V) of every node type in
    EMBED_SPLITS; for the rope builder also through hetero_pruned().live_ids32, whose target nodes are dead."""
    cfg, graph, (sc_d, vc_d) = _builder_features(name)
    g = _gen(31)
    for nt in sc_d:
        sc, vc = sc_d[nt].float().contiguous(), vc_d[nt].float().contiguous()
        S, V = sc.shape[1], vc.shape[1] // 3
        assert (S, V) in EMBED_SPLITS, f"{name} {nt}: (S, V) = {(S, V)} not among the tested splits"
        w = torch.randn(64, S + V, generator=g, device="cuda") / math.sqrt(S + V)
        g_x = torch.randn(sc.shape[0], 16, 64, generator=g, device="cuda")
        zero = (sc == 0).all(1) & (vc == 0).all(1)  # zero-padded object points
        _check_embed(f"embed {name} {nt}", sc, vc, w, g_x, cfg.ponita_dim, zero, perturb=False)
    if cfg.task != "rope":
        return
    pr = graph.hetero_pruned()
    assert [nt for nt in sc_d if nt not in pr.live_ids] == ["target_geometry"], "rope target nodes are not dead"
    for nt, ids in pr.live_ids32.items():
        sc, vc = sc_d[nt].float().clone(), vc_d[nt].float().clone()
        live = torch.zeros(sc.shape[0], dtype=torch.bool, device="cuda")
        live[ids.long()] = True
        sc[~live], vc[~live] = NAN, NAN
        S, V = sc.shape[1], vc.shape[1] // 3
        w = torch.randn(64, S + V, generator=g, device="cuda") / math.sqrt(S + V)
        g_x = torch.randn(ids.numel(), 16, 64, generator=g, device="cuda")
        _check_embed(f"embed {name} {nt} live rows", sc, vc, w, g_x, cfg.ponita_dim, node_ids=ids, counts=False,
                     perturb=False)
        _same_as_dense(sc, vc, w, g_x, cfg.ponita_dim, ids)


# ---------------------------------------------------------------------------------------------------------------------
# b. readout
# ---------------------------------------------------------------------------------------------------------------------
def _readout_desc(latent, w, b, od, odv, dim, **kw):
    from geometry_rl_b200 import _lib as L
    return L.GrlReadoutDesc(n_nodes=latent.shape[0], od=od, odv=odv, dim=dim, latent=L.ptr(latent), weight=L.ptr(w),
                            bias=L.ptr(b), ori=L.ptr(_ori(dim)),
                            **{k: L.ptr(v) if isinstance(v, torch.Tensor) else v for k, v in kw.items()})


def _readout_fwd(latent, w, b, od, odv, dim):
    from geometry_rl_b200 import _lib as L
    n = latent.shape[0]
    out = torch.full((n, odv, 3), NAN, device="cuda")
    hidden = torch.full((n, 64), NAN, device="cuda")
    L.call("grl_readout_fwd", C.byref(_readout_desc(latent, w, b, od, odv, dim, out=out, hidden=hidden)))
    return out, hidden


def _readout_bwd(latent, w, b, od, odv, dim, g_out, g_hid, n_p):
    """grad_latent and the partial slots [n_p, J * 64 + J] (gW | gb)."""
    from geometry_rl_b200 import _lib as L
    J = od + odv
    g_lat = torch.full_like(latent, NAN)
    part = torch.full((n_p, J * 64 + J), NAN, device="cuda")
    L.call("grl_readout_bwd", C.byref(_readout_desc(latent, w, b, od, odv, dim, grad_out=g_out, grad_hidden=g_hid,
                                                    grad_latent=g_lat, grad_partials=part, n_partials=n_p)))
    return g_lat, part


def _unpack_readout(part, J):
    g = part.double().sum(0)
    return g[:J * 64].view(J, 64), g[J * 64:]


def _readout_np(n):
    """ReadoutFn's partial count."""
    return max(1, min((n + 7) // 8, 2 * _sms()))


def _readout_inputs(n, od, odv, seed, scale=1.0, offset=0.0):
    """latent ~N(offset, scale); decoder weight ~N(0, 1/64), bias ~N(0, 0.5) (large enough for the bias term of the
    vector readout to matter); grad_out with a non-zero z, grad_hidden ~N(0, 1)."""
    g = _gen(seed)
    J = od + odv
    latent = torch.randn(n, 16, 64, generator=g, device="cuda") * scale + offset
    w = torch.randn(J, 64, generator=g, device="cuda") / 8
    b = torch.randn(J, generator=g, device="cuda") * 0.5
    g_out = torch.randn(n, odv, 3, generator=g, device="cuda")
    g_hid = torch.randn(n, 64, generator=g, device="cuda")
    return latent.contiguous(), w.contiguous(), b.contiguous(), g_out, g_hid


def _readout_ref(latent, w, b, od, odv, dim, g_out=None, g_hid=None):
    return ER.readout_reference(latent.to(D), w.to(D), b.to(D), _ori(dim).to(D), od, odv, dim,
                                None if g_out is None else g_out.to(D), None if g_hid is None else g_hid.to(D))


def _check_readout(tag, latent, w, b, od, odv, dim, g_out, g_hid, extra=0.0, counts=True, perturb=True):
    n, J = latent.shape[0], od + odv
    tol_hid, tol_out, tol_glat = TOL_HID + extra, TOL_OUT + extra, TOL_GLAT + extra
    n_p0 = _readout_np(n)
    out, hidden = _readout_fwd(latent, w, b, od, odv, dim)
    g_lat, part = _readout_bwd(latent, w, b, od, odv, dim, g_out, g_hid, n_p0)
    g_lat0, part0 = _readout_bwd(latent, w, b, od, odv, dim, g_out, None, n_p0)
    torch.cuda.synchronize()
    ref = _readout_ref(latent, w, b, od, odv, dim, g_out, g_hid)
    ref0 = _readout_ref(latent, w, b, od, odv, dim, g_out)
    bad, report = [], [f"n={n} od={od} odv={odv} dim={dim}"]
    _row(bad, report, "out", out.view(n, -1), ref["out"].view(n, -1), tol_out)
    _row(bad, report, "hidden", hidden, ref["hidden"], tol_hid)
    for g_l, p, r, what in ((g_lat, part, ref, "grad_hidden set"), (g_lat0, part0, ref0, "grad_hidden null")):
        _row(bad, report, f"{what}: grad_latent", g_l, r["grad"]["latent"], tol_glat)
        gw, gb = _unpack_readout(p, J)
        _glob(bad, report, f"{what}: grad W", gw, r["grad"]["weight"])
        _glob(bad, report, f"{what}: grad b", gb, r["grad"]["bias"])
    if dim == 2:
        assert torch.equal(out[..., 2], torch.zeros_like(out[..., 2])), "z of out is not exactly 0 in 2-D"
        gz = g_out.clone()
        gz[..., 2] = gz[..., 2] * -5.0 + 3.0
        g_latz, partz = _readout_bwd(latent, w, b, od, odv, dim, gz, g_hid, n_p0)
        assert torch.equal(g_latz, g_lat) and torch.equal(partz, part), "the z of grad_out reaches a gradient in 2-D"
    # exact: a second launch gives the same bits
    o2, h2 = _readout_fwd(latent, w, b, od, odv, dim)
    g2, p2 = _readout_bwd(latent, w, b, od, odv, dim, g_out, g_hid, n_p0)
    assert torch.equal(out, o2) and torch.equal(hidden, h2) and torch.equal(g_lat, g2) and torch.equal(part, p2), \
        "not repeatable"
    worst, n_blocks = 0.0, (n + 7) // 8
    gw0, gb0 = _unpack_readout(part, J)
    for n_p in sorted({1, n_blocks + 3} if counts else set()):
        g_l, p = _readout_bwd(latent, w, b, od, odv, dim, g_out, g_hid, n_p)
        assert torch.equal(g_l, g_lat), f"grad_latent depends on n_partials={n_p}"
        gw, gb = _unpack_readout(p, J)
        worst = max(worst, R.global_rel(gw, gw0), R.global_rel(gb, gb0))
        _glob(bad, [], f"n_partials={n_p} grad W", gw, ref["grad"]["weight"], REASSOC)
        _glob(bad, [], f"n_partials={n_p} grad b", gb, ref["grad"]["bias"], REASSOC)
        if n_p > n_blocks:
            assert torch.equal(p[n_blocks:], torch.zeros_like(p[n_blocks:])), f"n_partials={n_p}: idle slot not 0"
    if counts:
        report.append(f"partial counts: reassociation {worst:.3e} (tol {REASSOC:.0e})")
        if not worst < REASSOC:
            bad.append(f"partial counts move the decoder gradients by {worst:.3e}")
    _finish(tag, bad, report)
    if perturb:  # the last node: two orientation rows swapped (out), one orientation row dropped (hidden), the
        # upstream gradient of its first output vector dropped (grad_latent)
        sw = latent.clone()
        sw[n - 1, [2, 9]] = sw[n - 1, [9, 2]]
        r = R.row_rel(_readout_ref(sw, w, b, od, odv, dim)["out"].view(n, -1), ref["out"].view(n, -1))
        assert r >= 5 * tol_out, f"{tag}: two swapped orientation rows move out by {r:.3e} only"
        dr = latent.clone()
        dr[n - 1, 9] = 0
        r = R.row_rel(_readout_ref(dr, w, b, od, odv, dim)["hidden"], ref["hidden"])
        assert r >= 5 * tol_hid, f"{tag}: one dropped orientation row moves hidden by {r:.3e} only"
        go = g_out.clone()
        go[n - 1, 0] = 0
        r = R.row_rel(_readout_ref(latent, w, b, od, odv, dim, go, g_hid)["grad"]["latent"], ref["grad"]["latent"])
        assert r >= 5 * tol_glat, f"{tag}: one dropped upstream vector gradient moves grad_latent by {r:.3e} only"
    return ref


READOUT_OUTS = [(1, 1), (2, 2), (4, 4), (1, 3), (1, 7)]


def _readout_sizes():
    s = _sms()
    return [1, 7, 8, 9, 4 * s * 8 - 1, 4 * s * 8 + 1, 2 * s * 8 + 1, 16391]


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("od,odv", READOUT_OUTS, ids=[f"od{a}-odv{b}" for a, b in READOUT_OUTS])
def test_readout_kernels_alone_against_fp64(od, odv, dim):
    for n in _readout_sizes():
        latent, w, b, g_out, g_hid = _readout_inputs(n, od, odv, 100 * od + 10 * odv + dim + n)
        _check_readout(f"readout n={n} od={od} odv={odv} dim={dim}", latent, w, b, od, odv, dim, g_out, g_hid)


@pytest.mark.parametrize("case", ["offset", "1e-3", "1e3"])
@pytest.mark.parametrize("od,odv,dim", [(2, 2, 3), (1, 1, 2), (1, 7, 3)])
def test_readout_latent_scales(od, odv, dim, case):
    """Latent rows sharing a common offset of 30 over a unit spread (the vector readout's mean over orientations then
    cancels it), and latents at 1e-3 (the bias terms dominate) and 1e3 (they vanish)."""
    n = 4 * _sms() * 8 + 1
    offset, scale = (30.0, 1.0) if case == "offset" else (0.0, float(case))
    latent, w, b, g_out, g_hid = _readout_inputs(n, od, odv, 300 + dim, scale, offset)
    extra = (offset / scale) * OFFSET_ULPS * U
    _check_readout(f"readout {case} od={od} odv={odv} dim={dim}", latent, w, b, od, odv, dim, g_out, g_hid, extra,
                   counts=False, perturb=case == "offset")


@pytest.mark.parametrize("od,odv", [(5, 5), (1, 8)])
def test_readout_shapes_the_kernel_refuses(od, odv):
    """od + odv > GRL_READOUT_MAX_OUT: hepi.equivariant_readout runs the torch formulation, launches no readout
    kernel, and matches the fp64 reference forward and backward."""
    from geometry_rl_b200 import _lib as L
    from geometry_rl_b200.modules.pyg_models import hepi
    n, dim = 301, 3
    latent, w, b, g_out, g_hid = _readout_inputs(n, od, odv, 7)
    dec = torch.nn.Linear(64, od + odv).cuda()
    with torch.no_grad():
        dec.weight.copy_(w)
        dec.bias.copy_(b)
    x = latent.clone().requires_grad_(True)
    before = L.launch_count
    out, hidden = hepi.equivariant_readout(x, dec, _ori(dim)[:, :dim], od, odv, dim)
    ((out * g_out.view(-1, 3)).sum() + (hidden * g_hid).sum()).backward()
    torch.cuda.synchronize()
    assert L.launch_count == before, "a readout kernel was launched for a shape it refuses"
    ref = _readout_ref(latent, w, b, od, odv, dim, g_out, g_hid)
    bad, report = [], []
    _row(bad, report, "out", out.view(n, -1), ref["out"].view(n, -1), TOL_OUT)
    _row(bad, report, "hidden", hidden, ref["hidden"], TOL_HID)
    _row(bad, report, "grad_latent", x.grad, ref["grad"]["latent"], TOL_GLAT)
    _glob(bad, report, "grad W", dec.weight.grad, ref["grad"]["weight"])
    _glob(bad, report, "grad b", dec.bias.grad, ref["grad"]["bias"])
    _finish(f"readout torch formulation od={od} odv={odv}", bad, report)
