"""CPU: the fp64 references of tests/embed_readout_reference.py against the model's own formulations evaluated in fp32
(oracle.models.lift + F.linear for the embedding, hepi.equivariant_readout_torch for the readout), and every argument
check of grl_embed_fwd / _bwd and grl_readout_fwd / _bwd.  fp64 vs fp32 of the same operator: within 2e-5 of each
tensor's max magnitude, as tests/test_conv32_reference_cpu.py holds its references."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from oracle import models as om
from tests import conv16_reference as R
from tests import embed_readout_reference as ER

D = torch.float64
TOL = 2e-5
EINVAL, EUNSUPPORTED = -1, -2
LEGAL_OUTS = [(k, k) for k in range(1, 5)] + [(1, k) for k in range(2, 8)]  # od == odv or od == 1, od + odv <= 8


def _ori3(dim):
    ori = om.ori_grid(dim, 16, dim == 3)
    return torch.cat([ori, torch.zeros(16, 3 - dim)], 1)


def _bad(name, got, ref, bad):
    e = R.global_rel(got, ref)
    if not e < TOL:
        bad.append(f"{name} {e:.2e}")


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("S,V", [(1, 0), (0, 1), (3, 4), (7, 9), (16, 0)])
def test_embed_reference_matches_oracle_lift_fp32(S, V, dim):
    """x and the weight gradient; in 2-D the vectors carry a z the lift must not read; with node ids, rows of padded
    arrays (repeated, out of order) whose other rows are NaN."""
    gen = torch.Generator().manual_seed(11 * S + V + dim)
    n_pad, n = 23, 30
    sc = torch.randn(n_pad, S, generator=gen)
    vc = torch.randn(n_pad, 3 * V, generator=gen) * 2
    ids = torch.randint(0, n_pad - 5, (n,), generator=gen)
    ids[:3] = torch.tensor([7, 7, 2])
    sc[n_pad - 5:], vc[n_pad - 5:] = float("nan"), float("nan")
    w = (torch.randn(64, S + V, generator=gen) / (S + V) ** 0.5).requires_grad_(True)
    ori3 = _ori3(dim)
    g_x = torch.randn(n, 16, 64, generator=gen)
    x32 = F.linear(om.lift(sc[ids], vc[ids], ori3[:, :dim]), w)
    gw32, = torch.autograd.grad(x32, [w], g_x)
    ref = ER.embed_reference(sc.to(D), vc.to(D), w.detach().to(D), ori3.to(D), dim, ids.int(), grad_x=g_x.to(D))
    bad = []
    _bad("x", x32, ref["x"], bad)
    _bad("grad weight", gw32, ref["grad_weight"], bad)
    assert not bad, "\n".join(bad)
    if dim == 2 and V > 0:
        vz = vc.clone().view(n_pad, V, 3)
        vz[..., 2] += 5.0
        ref_z = ER.embed_reference(sc.to(D), vz.view(n_pad, 3 * V).to(D), w.detach().to(D), ori3.to(D), dim, ids)
        assert torch.equal(ref_z["x"], ref["x"]), "the z component reaches x in 2-D"


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("od,odv", LEGAL_OUTS)
def test_readout_reference_matches_hepi_torch_formulation_fp32(od, odv, dim):
    from geometry_rl_b200.modules.pyg_models import hepi
    gen = torch.Generator().manual_seed(100 * od + 10 * odv + dim)
    n = 13
    dec = torch.nn.Linear(64, od + odv)
    with torch.no_grad():
        dec.bias.normal_(0, 0.5, generator=gen)
    ori3 = _ori3(dim)
    latent = (torch.randn(n, 16, 64, generator=gen) + 0.3).requires_grad_(True)
    g_out = torch.randn(n, odv, 3, generator=gen)
    g_hid = torch.randn(n, 64, generator=gen)
    out32, hid32 = hepi.equivariant_readout_torch(latent, dec, ori3[:, :dim], od, odv, dim)
    g32 = torch.autograd.grad([out32, hid32], [latent, dec.weight, dec.bias], [g_out.reshape(-1, 3), g_hid])
    ref = ER.readout_reference(latent.detach().to(D), dec.weight.to(D), dec.bias.to(D), ori3.to(D), od, odv, dim,
                               grad_out=g_out.to(D), grad_hidden=g_hid.to(D))
    bad = []
    _bad("out", out32, ref["out"].reshape(-1, 3), bad)
    _bad("hidden", hid32, ref["hidden"], bad)
    for k, g in zip(("latent", "weight", "bias"), g32):
        _bad(f"grad {k}", g, ref["grad"][k], bad)
    assert not bad, "\n".join(bad)
    if dim == 2:
        assert torch.equal(ref["out"][..., 2], torch.zeros_like(ref["out"][..., 2])), "z of out is not 0 in 2-D"


@pytest.fixture(scope="module")
def lib():
    from geometry_rl_b200.csrc import build as b
    b.build()
    from geometry_rl_b200 import _lib
    return _lib


def _expect(lib, fn, d, code, msg):
    assert getattr(lib.load(), fn)(C.byref(d), None) == code, f"{fn}: {lib.last_error()}"
    assert msg in lib.last_error(), f"{fn}: {lib.last_error()!r} lacks {msg!r}"


def test_embed_rejects_invalid_arguments(lib):
    fake = 0x1000  # never dereferenced: every case fails validation before a launch

    def desc(**kw):
        base = dict(n_nodes=40, n_scalars=3, n_vectors=4, dim=3, scalars=fake, vectors=fake, ori=fake, weight=fake,
                    x=fake, grad_x=fake, grad_weight_partials=fake, n_partials=5)
        base.update(kw)
        return lib.GrlEmbedDesc(**base)

    for fn in ("grl_embed_fwd", "grl_embed_bwd"):
        _expect(lib, fn, desc(n_scalars=0, n_vectors=0), EUNSUPPORTED, "S+V=0 not in [1,16]")
        _expect(lib, fn, desc(n_scalars=9, n_vectors=8), EUNSUPPORTED, "S+V=17 not in [1,16]")
        _expect(lib, fn, desc(dim=4), EINVAL, "dim=4")
        _expect(lib, fn, desc(n_nodes=0), EINVAL, "n_nodes=0")
        _expect(lib, fn, desc(scalars=None), EINVAL, "null pointer")
        _expect(lib, fn, desc(vectors=None), EINVAL, "null pointer")
        assert getattr(lib.load(), fn)(None, None) == EINVAL
    _expect(lib, "grl_embed_fwd", desc(x=None), EINVAL, "grl_embed_fwd: null pointer")
    _expect(lib, "grl_embed_bwd", desc(n_partials=0), EINVAL, "n_partials=0")
    _expect(lib, "grl_embed_bwd", desc(grad_x=None), EINVAL, "grl_embed_bwd: null pointer")
    # S = 0 (V = 0) needs no scalar (vector) array
    for kw in (dict(n_scalars=0, scalars=None, dim=4), dict(n_vectors=0, vectors=None, dim=4)):
        _expect(lib, "grl_embed_fwd", desc(**kw), EINVAL, "dim=4")


def test_readout_rejects_invalid_arguments(lib):
    fake = 0x1000

    def desc(**kw):
        base = dict(n_nodes=40, od=2, odv=2, dim=3, latent=fake, weight=fake, bias=fake, ori=fake, out=fake,
                    hidden=fake, grad_out=fake, grad_hidden=None, grad_latent=fake, grad_partials=fake, n_partials=5)
        base.update(kw)
        return lib.GrlReadoutDesc(**base)

    for fn in ("grl_readout_fwd", "grl_readout_bwd"):
        _expect(lib, fn, desc(od=2, odv=3), EUNSUPPORTED, "od=2 odv=3")
        _expect(lib, fn, desc(od=1, odv=8), EUNSUPPORTED, "od=1 odv=8")
        _expect(lib, fn, desc(od=5, odv=4), EUNSUPPORTED, "od=5 odv=4")
        _expect(lib, fn, desc(od=0, odv=1), EUNSUPPORTED, "od=0 odv=1")
        _expect(lib, fn, desc(dim=4), EINVAL, "dim=4")
        _expect(lib, fn, desc(n_nodes=0), EINVAL, "n_nodes=0")
        _expect(lib, fn, desc(latent=None), EINVAL, "null pointer")
        assert getattr(lib.load(), fn)(None, None) == EINVAL
    _expect(lib, "grl_readout_fwd", desc(hidden=None), EINVAL, "null output pointer")
    _expect(lib, "grl_readout_bwd", desc(grad_out=None), EINVAL, "null grad pointer")
    _expect(lib, "grl_readout_bwd", desc(grad_partials=None), EINVAL, "null grad pointer")
    _expect(lib, "grl_readout_bwd", desc(n_partials=0), EINVAL, "n_partials=0")
