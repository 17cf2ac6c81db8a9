"""CPU: the observation-normalisation kernels' (csrc/grl_obsnorm.cu) slot split restated in numpy, the GrlVecNormDesc
mirror against the C compiler, the argument checks through the C ABI (they return before any launch), ops.vecnorm's
refusal of CPU tensors, and NDVecNorm.load_state_dict restoring into the existing state tensors."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "grl_b200.h")
ROWS_PER_SLOT, MAX_SLOTS = 512, 1024


def slots(M):
    """S(M) of grl_vecnorm_stats: max(1, min(ceil(M / 512), 1024))."""
    return max(1, min(-(-M // ROWS_PER_SLOT), MAX_SLOTS))


def slot_ranges(M):
    """Rows [lo, hi) of each slot: P = ceil(M / S) rows per slot, clamped to M."""
    S = slots(M)
    P = -(-M // S) if M else 0
    s = np.arange(S, dtype=np.int64)
    lo = np.minimum(s * P, M)
    return lo, np.minimum(lo + P, M)


@pytest.mark.parametrize("M", [0, 1, 2, 511, 512, 513, 1025, 4096 * 97, 4096 * 4, 1000 * 97, 200 * 162, 100 * 460,
                               MAX_SLOTS * ROWS_PER_SLOT, MAX_SLOTS * ROWS_PER_SLOT + 1, 3 * MAX_SLOTS * ROWS_PER_SLOT + 7])
def test_every_row_is_counted_once(M):
    lo, hi = slot_ranges(M)
    assert 1 <= len(lo) <= MAX_SLOTS
    cover = np.zeros(M + 1, dtype=np.int64)
    for a, b in zip(lo, hi):
        assert 0 <= a <= b <= M
        cover[a:b] += 1
    assert (cover[:M] == 1).all()
    # slots are contiguous and in row order: the fixed-order sum over slots is a sum in row-block order
    assert (lo[1:] == hi[:-1]).all() and lo[0] == 0 and hi[-1] == M


def test_split_depends_on_the_rows_only():
    """The host's slot count is the restated one, and neither changes with the SM count or an SM reservation."""
    from geometry_rl_b200 import _lib as L, ops
    assert (L.VECNORM_ROWS_PER_SLOT, L.VECNORM_MAX_SLOTS) == (ROWS_PER_SLOT, MAX_SLOTS)
    Ms = [0, 1, 97, 513, 4096 * 97, 10 ** 7]
    before = [ops.vecnorm_slots(M) for M in Ms]
    L.reserve_sms(4)
    try:
        assert [ops.vecnorm_slots(M) for M in Ms] == before
    finally:
        L.reserve_sms(0)
    assert before == [slots(M) for M in Ms]
    # slots grow with M until the cap: the grid scales with the rollout's row count
    assert slots(4096 * 97) == 776 and slots(4096 * 4) == 32 and slots(1) == 1


@pytest.fixture(scope="module")
def lib():
    from geometry_rl_b200.csrc import build as b
    b.build()
    from geometry_rl_b200 import _lib
    return _lib


def test_vecnorm_desc_layout_matches_the_c_compiler(lib):
    structs = {"GrlVecNormKey": lib.GrlVecNormKey, "GrlVecNormDesc": lib.GrlVecNormDesc}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void) {"]
    for name, cls in structs.items():
        lines.append(f'printf("{name} %zu\\n", sizeof({name}));')
        lines += [f'printf("{name}.{f} %zu\\n", offsetof({name}, {f}));' for f, _ in cls._fields_]
    for m in ("GRL_VECNORM_MAX_KEYS", "GRL_VECNORM_MAX_COMPS", "GRL_VECNORM_ROWS_PER_SLOT", "GRL_VECNORM_MAX_SLOTS"):
        lines.append(f'printf("{m} %d\\n", {m});')
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
    assert int(layout["GRL_VECNORM_MAX_KEYS"]) == lib.VECNORM_MAX_KEYS
    assert int(layout["GRL_VECNORM_MAX_COMPS"]) == lib.VECNORM_MAX_COMPS
    assert int(layout["GRL_VECNORM_ROWS_PER_SLOT"]) == lib.VECNORM_ROWS_PER_SLOT
    assert int(layout["GRL_VECNORM_MAX_SLOTS"]) == lib.VECNORM_MAX_SLOTS


def test_vecnorm_rejects_invalid_arguments(lib):
    handle = lib.load()
    fake = 0x1000  # never dereferenced: every case fails validation before a launch
    EINVAL, EUNSUPPORTED = -1, -2

    def desc(n_keys=2, partials=fake, inc=fake, world=1, **key):
        d = lib.GrlVecNormDesc(n_keys=n_keys, world=world, decay=0.9999, eps=1e-4, partials=partials, inc=inc)
        for i in range(2):
            base = dict(batch=4, feat=291, comps=3, x=fake, out=fake, sum=fake, ssq=fake, count=fake)
            if i == 1:
                base.update(key)
            d.key[i] = lib.GrlVecNormKey(**base)
        return d

    entries = ("grl_vecnorm_stats", "grl_vecnorm_update", "grl_vecnorm_apply")
    everywhere = [desc(comps=0), desc(feat=290), desc(batch=-1), desc(feat=-3), desc(n_keys=0), desc(n_keys=9),
                  desc(world=0)]
    for fn in entries:
        for d in everywhere:
            assert getattr(handle, fn)(C.byref(d), None) == EINVAL, f"{fn}: {lib.last_error()}"
        assert getattr(handle, fn)(C.byref(desc(comps=65, feat=65)), None) == EUNSUPPORTED, lib.last_error()
        assert getattr(handle, fn)(None, None) == EINVAL
    handle.grl_vecnorm_apply(C.byref(desc(comps=0)), None)
    assert "comps=0" in lib.last_error()
    handle.grl_vecnorm_apply(C.byref(desc(feat=290)), None)
    assert "not a multiple" in lib.last_error()
    # each entry point needs its own pointers
    for d in (desc(x=None), desc(partials=None), desc(inc=None)):
        assert handle.grl_vecnorm_stats(C.byref(d), None) == EINVAL, lib.last_error()
    for d in (desc(inc=None), desc(sum=None), desc(ssq=None), desc(count=None)):
        assert handle.grl_vecnorm_update(C.byref(d), None) == EINVAL, lib.last_error()
    for d in (desc(x=None), desc(out=None), desc(sum=None), desc(count=None)):
        assert handle.grl_vecnorm_apply(C.byref(d), None) == EINVAL, lib.last_error()


def test_vecnorm_refuses_cpu_tensors():
    from geometry_rl_b200 import ops
    x = torch.zeros(4, 9)
    z = lambda: torch.zeros(3)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.vecnorm([x], out=[torch.empty_like(x)], sums=[z()], ssqs=[z()], counts=[torch.zeros(1)], decay=0.9999,
                    eps=1e-4)
    from geometry_rl_b200.torchrl.envs import NDVecNorm
    norm = NDVecNorm(in_keys=["position_vectors"], out_keys=["norm_position_vectors"], shapes=[3])
    with pytest.raises(RuntimeError, match="CUDA"):
        norm.apply_device({"position_vectors": x})


def test_load_state_dict_restores_into_the_existing_tensors():
    from geometry_rl_b200.torchrl.envs import NDVecNorm
    g = torch.Generator().manual_seed(0)
    norm = NDVecNorm(in_keys=["position_vectors"], out_keys=["norm_position_vectors"], shapes=[3], decay=0.999)
    norm({"position_vectors": torch.randn(4, 5, 3, generator=g)})
    sd = norm.state_dict()
    held = dict(norm._stats["position_vectors"])
    norm({"position_vectors": torch.randn(4, 5, 3, generator=g)})
    assert not torch.equal(held["sum"], sd["position_vectors_sum"])
    norm.load_state_dict(sd)
    for n, t in norm._stats["position_vectors"].items():
        assert t is held[n] and torch.equal(t, sd[f"position_vectors_{n}"])
    # a fresh normaliser takes clones
    other = NDVecNorm(in_keys=["position_vectors"], out_keys=["norm_position_vectors"], shapes=[3])
    other.load_state_dict(sd)
    assert other._stats["position_vectors"]["sum"] is not sd["position_vectors_sum"]
    assert torch.equal(other._stats["position_vectors"]["sum"], sd["position_vectors_sum"])
