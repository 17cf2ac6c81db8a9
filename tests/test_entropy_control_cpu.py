"""CPU: TRPL entropy control on the fused path.  The fp64 restatement of both entropy schedules (the formula
grl_trpl_entropy_bound evaluates) against the torch schedules of projection_utils.py, the descriptor layouts against
the C compiler, and the argument checks of grl_trpl_entropy_bound and of the entropy fields of grl_trpl_fwd / _bwd."""
import ctypes as C
import os
import subprocess
import tempfile

import pytest
import torch

from tests import entropy_reference as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "grl_b200.h")
EINVAL, EUNSUPPORTED = -1, -2


@pytest.mark.parametrize("kind", ["linear", "exp"])
@pytest.mark.parametrize("k", [3, 6, 12])
def test_schedule_restatement_matches_the_torch_schedule(kind, k):
    from geometry_rl_b200.algorithms.trust_region_projections.utils.projection_utils import get_entropy_schedule
    T = 1000
    f = get_entropy_schedule(kind, T, dim=k)
    for ie, te, temp in ((1.42 * k, -0.5, 0.5), (-2.0, 1.5, 0.9), (0.3, 0.3, 2.0)):
        for step in (0, 1, 7, 250, 999, 1000, 1500):
            ref = f(torch.tensor(ie, dtype=torch.float64), torch.tensor(te, dtype=torch.float64), temp, step)
            got = R.schedule(kind, ie, te, temp, step, T, k)
            assert abs(float(ref) - float(got)) <= 1e-12 * max(1.0, abs(float(ref))), (ie, te, temp, step)
    # linear does not scale the target by k (projection_utils.py:41-47): at step T the bound is te itself
    assert R.schedule("linear", 5.0, -1.0, 0.5, T, T, k) == -1.0
    assert abs(R.schedule("exp", 5.0, -1.0, 0.5, 0, T, k) - 5.0) < 1e-12


@pytest.fixture(scope="module")
def lib():
    from geometry_rl_b200.csrc import build as b
    b.build()
    from geometry_rl_b200 import _lib
    return _lib


def test_descriptor_layouts_and_constants_match_the_c_compiler(lib):
    structs = {"GrlProjDesc": lib.GrlProjDesc, "GrlEntropyBoundDesc": lib.GrlEntropyBoundDesc}
    macros = ("GRL_ENTROPY_OFF", "GRL_ENTROPY_INEQ", "GRL_ENTROPY_EQ", "GRL_ENTROPY_LINEAR", "GRL_ENTROPY_EXP")
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void) {"]
    for name, cls in structs.items():
        lines.append(f'printf("{name} %zu\\n", sizeof({name}));')
        lines += [f'printf("{name}.{f} %zu\\n", offsetof({name}, {f}));' for f, _ in cls._fields_]
    lines += [f'printf("{m} %d\\n", {m});' for m in macros]
    lines += ["return 0; }"]
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "t.c"), os.path.join(d, "t")
        open(src, "w").write("\n".join(lines))
        subprocess.run(["gcc", src, "-o", exe], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    layout = dict(l.split() for l in out.strip().splitlines())
    for name, cls in structs.items():
        assert int(layout[name]) == C.sizeof(cls), name
        for f, _ in cls._fields_:
            assert int(layout[f"{name}.{f}"]) == getattr(cls, f).offset, f"{name}.{f}"
    assert lib.ENTROPY_MODE == {"ineq": int(layout["GRL_ENTROPY_INEQ"]), "eq": int(layout["GRL_ENTROPY_EQ"])}
    assert int(layout["GRL_ENTROPY_OFF"]) == 0
    assert lib.ENTROPY_SCHEDULE == {"linear": int(layout["GRL_ENTROPY_LINEAR"]), "exp": int(layout["GRL_ENTROPY_EXP"])}


def test_entropy_bound_rejects_invalid_arguments(lib):
    handle = lib.load()
    fake = 0x1000  # never dereferenced: every case fails validation before a launch

    def desc(**kw):
        base = dict(batch=8, k=6, schedule=1, stage=0, total_train_steps=1000, target_entropy=0.0, temperature=0.5,
                    old_v=fake, step=fake, sums=fake, state=fake)
        base.update(kw)
        return lib.GrlEntropyBoundDesc(**base)

    cases = [(desc(schedule=0), EUNSUPPORTED, "schedule=0"), (desc(schedule=3), EUNSUPPORTED, "schedule=3"),
             (desc(total_train_steps=0), EINVAL, "total_train_steps=0"),
             (desc(total_train_steps=-5), EINVAL, "total_train_steps=-5"),
             (desc(schedule=2, temperature=0.0), EINVAL, "temperature"),
             (desc(schedule=2, temperature=-0.5), EINVAL, "temperature"),
             (desc(batch=0), EINVAL, "batch=0"), (desc(k=17), EUNSUPPORTED, "k=17"), (desc(stage=3), EINVAL, "stage=3"),
             (desc(old_v=None), EINVAL, "null"), (desc(step=None), EINVAL, "null"), (desc(sums=None), EINVAL, "null"),
             (desc(state=None), EINVAL, "null"), (desc(stage=1, old_v=None), EINVAL, "null")]
    for d, code, msg in cases:
        assert handle.grl_trpl_entropy_bound(C.byref(d), None) == code, lib.last_error()
        assert msg in lib.last_error()
    assert handle.grl_trpl_entropy_bound(None, None) == EINVAL
    # linear ignores the temperature: this one fails on the null state only
    assert handle.grl_trpl_entropy_bound(C.byref(desc(temperature=0.0, state=None)), None) == EINVAL
    assert "null" in lib.last_error()


def test_projection_rejects_inconsistent_entropy_fields(lib):
    handle = lib.load()
    fake = 0x1000

    def desc(**kw):
        base = dict(batch=8, k=6, proj_type=0, eps_mean=0.05, eps_cov=0.01, mean=fake, v=fake, old_mean=fake, old_v=fake,
                    proj_mean=fake, proj_v=fake, eta=fake, grad_proj_mean=fake, grad_proj_v=fake, grad_mean=fake,
                    grad_v=fake, entropy_mode=1, entropy_first=0, entropy_beta=fake, entropy_alpha=fake)
        base.update(kw)
        return lib.GrlProjDesc(**base)

    for fn in ("grl_trpl_fwd", "grl_trpl_bwd"):
        for d, code in ((desc(entropy_mode=3), EUNSUPPORTED), (desc(entropy_mode=-1), EUNSUPPORTED),
                        (desc(entropy_mode=0, entropy_first=1), EINVAL), (desc(entropy_first=2), EINVAL),
                        (desc(entropy_alpha=None), EINVAL)):
            assert getattr(handle, fn)(C.byref(d), None) == code, f"{fn}: {lib.last_error()}"
    assert handle.grl_trpl_fwd(C.byref(desc(entropy_beta=None)), None) == EINVAL
    assert "entropy" in lib.last_error()
    # the backward of the projection-after mode reads the final proj_v
    assert handle.grl_trpl_bwd(C.byref(desc(proj_v=None)), None) == EINVAL
    assert "proj_v" in lib.last_error()


def test_build_agent_passes_projection_keywords_through():
    from geometry_rl_b200 import learner
    from geometry_rl_b200.synthetic import CONFIGS
    cfg = CONFIGS["rope_shaping_hepi_trpl_cfg"]
    _, _, pr, loss_module, _ = learner.build_agent(cfg, "cpu", projection_kwargs=dict(
        entropy_schedule="exp", target_entropy=-1.5, temperature=0.7, entropy_eq=True, entropy_first=True,
        total_train_steps=40))
    assert pr.has_entropy_control and pr.entropy_eq and pr.entropy_first and pr.total_train_steps == 40
    assert pr.temperature == 0.7 and float(pr.target_entropy) == -1.5
    assert loss_module.projection is pr and pr.entropy_bound is None
    _, _, pr0, _, _ = learner.build_agent(cfg, "cpu")
    assert not pr0.has_entropy_control
