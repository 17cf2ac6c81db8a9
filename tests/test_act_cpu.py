"""CPU: the numpy reference of the acting noise (tests/philox_reference.py) against the Random123 known-answer vectors and
the documented Box-Muller mapping; the GrlActDesc mirror against the C compiler; grl_gaussian_act's argument checks,
which return before any launch (no GPU here)."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

from tests import philox_reference as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "grl_b200.h")

# Random123 kat_vectors, philox4x32 with 10 rounds: (counter, key, output)
KAT = [
    ((0x00000000, 0x00000000, 0x00000000, 0x00000000), (0x00000000, 0x00000000),
     (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff), (0xffffffff, 0xffffffff),
     (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


def test_philox_matches_random123_known_answers():
    ctr = np.array([c for c, _, _ in KAT], dtype=np.uint64)
    key = np.array([k for _, k, _ in KAT], dtype=np.uint64)
    out = P.philox4x32_10(ctr, key)
    assert out.tolist() == [list(o) for _, _, o in KAT]


def test_box_muller_mapping_as_documented():
    # the extreme words map strictly inside (0, 1): no log(0), and the largest radius is sqrt(2 * 33 ln 2)
    u = P.uniform(np.array([0, 0xFFFFFFFF], dtype=np.uint64))
    assert u[0] == 2.0 ** -33 and u[1] == 1.0 - 2.0 ** -33 and 0.0 < u[0] < u[1] < 1.0
    # component c of sample s at state {seed, call}: block c // 4 of counter (c // 4, s, call lo, call hi), key
    # (seed lo, seed hi ^ rank); components 2m, 2m+1 share the pair (u_2m', u_2m'+1) of the block as cos / sin
    seed, call, rank, s, c = 0x123456789ABCDEF0, (7 << 32) + 5, 3, 11, 6
    w = P.philox4x32_10(np.array([c // 4, s, call & P.MASK, call >> 32], dtype=np.uint64),
                        np.array([seed & P.MASK, (seed >> 32) ^ rank], dtype=np.uint64))
    u = (w.astype(np.float64) + 0.5) / 2.0 ** 32
    expect = math.sqrt(-2.0 * math.log(u[2])) * math.cos(2.0 * math.pi * u[3])  # c % 4 == 2 -> pair 1, cos
    eps = P.act_eps(seed, call, 16, 9, rank=rank)
    assert eps.dtype == np.float32 and eps.shape == (16, 9)
    assert eps[s, c] == np.float32(expect)
    assert eps[s, c + 1] == np.float32(math.sqrt(-2.0 * math.log(u[2])) * math.sin(2.0 * math.pi * u[3]))
    # a component's draw does not depend on k (nor on the batch size)
    assert np.array_equal(P.act_eps(seed, call, 12, 32, rank=rank)[:, :9], eps[:12])
    # rank 0 keys on the seed alone; other ranks, calls and seeds give other draws
    assert not np.array_equal(P.act_eps(seed, call, 16, 9, rank=0), eps)
    assert not np.array_equal(P.act_eps(seed, call + 1, 16, 9, rank=rank), eps)
    assert not np.array_equal(P.act_eps(seed + 1, call, 16, 9, rank=rank), eps)


def test_reference_draws_look_standard_normal():
    from scipy import stats
    z = P.act_eps(2024, 0, 1 << 14, 32).astype(np.float64).reshape(-1)
    assert stats.kstest(z, "norm").pvalue > 1e-3
    assert abs(z.mean()) < 5e-3 and abs(z.std() - 1.0) < 5e-3


@pytest.fixture(scope="module")
def lib():
    from geometry_rl_b200.csrc import build as b
    b.build()
    from geometry_rl_b200 import _lib
    return _lib


def test_act_desc_layout_matches_the_c_compiler(lib):
    cls = lib.GrlActDesc
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void) {",
             'printf("size %zu\\n", sizeof(GrlActDesc));']
    lines += [f'printf("{f} %zu\\n", offsetof(GrlActDesc, {f}));' for f, _ in cls._fields_]
    lines += ['printf("max_k %d\\n", GRL_ACT_MAX_K);', "return 0; }"]
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "t.c"), os.path.join(d, "t")
        open(src, "w").write("\n".join(lines))
        subprocess.run(["gcc", src, "-o", exe], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    layout = dict(l.split() for l in out.strip().splitlines())
    assert int(layout["size"]) == C.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(layout[f]) == getattr(cls, f).offset, f
    assert int(layout["max_k"]) == lib.ACT_MAX_K


def test_gaussian_act_rejects_unsupported_shapes_and_null_pointers(lib):
    handle = lib.load()
    fake = 0x1000  # never dereferenced: every case fails validation before a launch

    def desc(**kw):
        base = dict(batch=4, num_rows=2, action_dim=3, hidden_dim=64, post_fc=1, contextual_std=1, hidden=fake,
                    mean_weight=fake, mean_bias=fake, std_weight=fake, std_bias=fake, state=fake, loc=fake, cov=fake,
                    action=fake, log_prob=fake)
        base.update(kw)
        return lib.GrlActDesc(**base)

    unsupported = [desc(hidden_dim=32), desc(num_rows=4, action_dim=9), desc(num_rows=33, action_dim=1)]
    invalid = [desc(batch=0), desc(state=None), desc(cov=None), desc(hidden=None), desc(post_fc=0, mean=None),
               desc(contextual_std=1, std_bias=None), desc(std_weight=None)]
    for d in unsupported:
        assert handle.grl_gaussian_act(C.byref(d), None) == -2, lib.last_error()
    for d in invalid:
        assert handle.grl_gaussian_act(C.byref(d), None) == -1, lib.last_error()
    assert handle.grl_act_advance(None, None) == -1


def test_data_parallel_attach_gives_the_actor_its_rank():
    """Under data parallelism the rank enters the acting noise's key (PolicyOperator.act_rank), with no collective."""
    import torch
    from geometry_rl_b200 import ops
    from geometry_rl_b200.parallel import DataParallel

    class _Loss:
        actor_network = torch.nn.Module()
        critic_network = torch.nn.Module()

    dp = DataParallel.__new__(DataParallel)  # a rank's view without a process group: attach issues no collective
    dp.rank, dp.world_size, dp.side, dp.collectives = 3, 4, None, 0
    try:
        dp.attach(_Loss)
    finally:
        ops.set_calibration_std(None)
    assert _Loss.actor_network.act_rank == 3 and dp.collectives == 0
