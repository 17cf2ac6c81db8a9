"""CPU: the fp64 references of tests/conv32_reference.py against `oracle.models` evaluated in fp32 the way the models
call it.  fp64 vs fp32 of the same operator, so the difference is fp32 rounding alone: within 2e-5 of each tensor's max
magnitude, as tests/test_conv_reference_cpu.py holds the layer reference."""
import pytest
import torch

from oracle import models as om
from tests import conv16_reference as R
from tests import conv32_reference as R32
from tests.conv16_reference import random_params

D = torch.float64
TOL = 2e-5


def _ori3(dim):
    ori = om.ori_grid(dim, 16)
    return torch.cat([ori, torch.zeros(16, 3 - dim)], 1)


def _bad(name, got, ref, bad):
    e = R.global_rel(got, ref)
    if not e < TOL:
        bad.append(f"{name} {e:.2e}")


@pytest.mark.parametrize("dim", [2, 3])
def test_basis_reference_matches_oracle_fp32(dim):
    """The basis and its four weight gradients, with coincident endpoints (a zero relative vector) among the edges."""
    gen = torch.Generator().manual_seed(31 + dim)
    p = {k: v.requires_grad_(True) for k, v in random_params(gen).items()}
    n, E = 17, 60
    pos_src = torch.randn(n, 3, generator=gen) * 0.7
    pos_dst = torch.randn(n, 3, generator=gen) * 0.7
    ei = torch.stack([torch.randint(0, n, (E,), generator=gen), torch.randint(0, n, (E,), generator=gen)])
    pos_dst[ei[1, :5]] = pos_src[ei[0, :5]]  # coincident endpoints
    ori3 = _ori3(dim)
    sp, _ = om.invariants(ori3[:, :dim], pos_src[ei[0]][:, :dim], pos_dst[ei[1]][:, :dim])
    assert bool((sp[:5].abs().amax((1, 2)) == 0).any()), "no edge with a zero relative vector"
    sd = {"basis_fn.1.weight": p["bw1"], "basis_fn.1.bias": p["bb1"], "basis_fn.3.weight": p["bw2"],
          "basis_fn.3.bias": p["bb2"]}
    basis32 = om.basis_mlp(sp, sd, "basis_fn")
    g_basis = torch.randn(E, 16, 64, generator=gen)
    g32 = torch.autograd.grad(basis32, [p[k] for k in R32.BASIS], g_basis)
    ref = R32.basis_reference(pos_src.to(D), pos_dst.to(D), p, ori3.to(D), dim, ei, grad_basis=g_basis.to(D))
    bad = []
    _bad("basis", basis32, ref["basis"], bad)
    for k, g in zip(R32.BASIS, g32):
        _bad(f"grad {k}", g, ref["grad"][k], bad)
    assert not bad, "\n".join(bad)


def test_spatial_reference_matches_oracle_fp32():
    gen = torch.Generator().manual_seed(41)
    n_src, n_dst, E = 11, 6, 50
    x_src = torch.randn(n_src, 16, 64, generator=gen).requires_grad_(True)
    basis = torch.randn(E, 16, 64, generator=gen).requires_grad_(True)
    wk = (torch.randn(64, 64, generator=gen) * 0.12).requires_grad_(True)
    ei = torch.stack([torch.randint(0, n_src, (E,), generator=gen), torch.randint(0, n_dst - 1, (E,), generator=gen)])
    kern = torch.nn.functional.linear(basis, wk)
    x1 = torch.zeros(n_dst, 16, 64).index_add_(0, ei[1], kern * x_src[ei[0]])
    g_x1 = torch.randn(n_dst, 16, 64, generator=gen)
    g32 = torch.autograd.grad(x1, [x_src, basis, wk], g_x1)
    ref = R32.spatial_reference(x_src.to(D), basis.to(D), wk.to(D), ei, n_dst, grad_x1=g_x1.to(D))
    bad = []
    _bad("x1", x1, ref["x1"], bad)
    for k, g in zip(("x_src", "basis", "wk"), g32):
        _bad(f"grad {k}", g, ref["grad"][k], bad)
    assert not bad, "\n".join(bad)
    assert bool((ref["x1"][n_dst - 1] == 0).all()), "a node without in-edges has x1 = 0"


def test_node_reference_matches_oracle_fp32():
    """The identity-message node reference against the oracle's fibre convolution + ConvNeXt update fed x1 directly."""
    gen = torch.Generator().manual_seed(43)
    p = {k: v.requires_grad_(True) for k, v in random_params(gen).items()}
    n = 9
    x1 = torch.randn(n, 16, 64, generator=gen).requires_grad_(True)
    x_dst = torch.randn(n, 16, 64, generator=gen)
    x1.data[3] = 0  # a node without in-edges
    g_out = torch.randn(n, 16, 64, generator=gen)
    sd = {"c.bias": p["bias"], "m.0.weight": p["ln_g"], "m.0.bias": p["ln_b"], "m.1.weight": p["w1"],
          "m.1.bias": p["b1"], "m.3.weight": p["w2"], "m.3.bias": p["b2"]}
    x2 = torch.einsum("boc,opc->bpc", x1, p["fk"]) / 16 + p["bias"]
    out = om.convnext_update(x_dst, x2, sd, "m.0", "m.1", "m.3")
    names = ["fk", "bias", "ln_g", "ln_b", "w1", "b1", "w2", "b2"]
    g32 = torch.autograd.grad(out, [x1] + [p[k] for k in names], g_out)
    ref = R32.node_reference(x1.detach().to(D), x_dst.to(D), {k: v.detach().to(D) for k, v in p.items()},
                             grad_out=g_out.to(D))
    bad = []
    _bad("out", out, ref["out"], bad)
    _bad("x2", x2, ref["x2"], bad)
    for k, g in zip(["x_src"] + names, g32):
        _bad(f"grad {k}", g, ref["grad"][k], bad)
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("flavour", ["hepi", "empn"])
def test_calibration_reference_matches_oracle_fp32(flavour):
    """The factors from the oracle's own intermediates (fiber_bundle_conv's x1 and x2 - bias), as
    test_calibration_matches_reference_semantics derives them; EMPN's fibre kernel is [p][o][c] in the oracle
    (fiber_transposed) and [o][p][c] in the calibration, as ponita.py passes it."""
    gen = torch.Generator().manual_seed(47)
    p = random_params(gen)
    n_src, n_dst, E = 15, 15, 70
    x_src = torch.randn(n_src, 16, 64, generator=gen)
    x_dst = x_src if flavour == "empn" else torch.randn(n_dst, 16, 64, generator=gen) * 1.3
    pos = torch.randn(n_src, 3, generator=gen) * 0.7
    ei = torch.stack([torch.randint(0, n_src, (E,), generator=gen), torch.randint(0, n_dst, (E,), generator=gen)])
    ori3 = _ori3(3)
    sp, _ = om.invariants(ori3, pos[ei[0]], pos[ei[1]])
    sd = {"basis_fn.1.weight": p["bw1"], "basis_fn.1.bias": p["bb1"], "basis_fn.3.weight": p["bw2"],
          "basis_fn.3.bias": p["bb2"], "c.kernel.weight": p["wk"], "c.fiber_kernel.weight": torch.eye(64),
          "c.bias": p["bias"]}
    kb = om.basis_mlp(sp, sd, "basis_fn")
    fk_op = p["fk"]  # [o][p][c], the kernels' layout
    fb = fk_op.transpose(0, 1).contiguous() if flavour == "empn" else fk_op
    inter = {}
    x2 = om.fiber_bundle_conv(x_src, x_dst, ei, kb, fb, sd, "c", fiber_transposed=flavour == "empn",
                              intermediates=inter) - p["bias"]
    f1, f2 = x_dst.std() / inter["x1"].std(), inter["x1"].std() / x2.std()
    basis = R32.basis_reference(pos.to(D), pos.to(D), p, ori3.to(D), 3, ei)["basis"]
    x1 = R32.spatial_reference(x_src.to(D), basis, p["wk"].to(D), ei, n_dst)["x1"]
    r1, r2 = R32.calibration_reference(x_dst.to(D), x1, fk_op.to(D))
    assert abs(float(f1) / float(r1) - 1) < TOL and abs(float(f2) / float(r2) - 1) < TOL, (f1, r1, f2, r2)
