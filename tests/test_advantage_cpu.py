"""CPU: the grouped work split of grl_critic_inner_stats / _fwd (per-time-step statistics of the advantage phase) restated
in numpy and checked against the single-group split it extends; the host's choice of slots per group; the argument checks
of the four critic entry points for `n_groups`, through the C ABI without a device."""
import ctypes as C

import numpy as np
import pytest


def single_group_range(n_graphs, n_partials):
    """The split of the graphs over the grid before groups existed (one group): CTA c -> [lo, hi)."""
    c = np.arange(n_partials, dtype=np.int64)
    return n_graphs * c // n_partials, n_graphs * (c + 1) // n_partials


def grouped_range(n_graphs, n_partials, n_groups):
    """critic_range of csrc/grl_critic.cu: S = n_partials / n_groups slots per group, CTA c serves group c / S, slot c % S."""
    S, bg = n_partials // n_groups, n_graphs // n_groups
    c = np.arange(n_partials, dtype=np.int64)
    g, s = c // S, c % S
    return g * bg + bg * s // S, g * bg + bg * (s + 1) // S, g


def host_slots(n_graphs, n_groups, sm_count):
    """ops.CriticInnerFn: slots per group for n_groups > 1."""
    bg = n_graphs // n_groups
    return max(1, min(bg, -(-2 * sm_count // n_groups)))


@pytest.mark.parametrize("n_graphs,n_partials", [(1, 1), (7, 3), (97, 96), (8192, 296), (101000, 296), (300, 300)])
def test_one_group_is_the_single_group_split(n_graphs, n_partials):
    lo, hi, g = grouped_range(n_graphs, n_partials, 1)
    lo1, hi1 = single_group_range(n_graphs, n_partials)
    assert np.array_equal(lo, lo1) and np.array_equal(hi, hi1) and not g.any()


@pytest.mark.parametrize("b_env,groups", [(1000, 101), (100, 101), (4096, 17), (200, 201), (1, 2), (2, 300), (1, 301),
                                          (256, 33), (5, 12), (37, 3)])
@pytest.mark.parametrize("sm_count", [148, 144])
def test_grouped_split_covers_every_graph_once_within_its_group(b_env, groups, sm_count):
    n_graphs = b_env * groups
    S = host_slots(n_graphs, groups, sm_count)
    assert 1 <= S <= b_env
    lo, hi, g = grouped_range(n_graphs, groups * S, groups)
    cover = np.zeros(n_graphs, dtype=np.int64)
    for a, b in zip(lo, hi):
        cover[a:b] += 1
    assert (cover == 1).all()
    # a CTA never spans two groups, and group g's CTAs are contiguous slots g*S .. g*S + S-1
    assert (lo >= g * b_env).all() and (hi <= (g + 1) * b_env).all()
    assert np.array_equal(g, np.repeat(np.arange(groups), S))
    # every CTA has work unless a group has fewer graphs than slots (never: S <= Bg)
    assert (hi > lo).all()


@pytest.mark.parametrize("b_env,groups", [(1000, 101), (100, 101), (4096, 17), (200, 201), (1, 2), (2, 300), (64, 1)])
def test_host_picks_the_documented_slots(b_env, groups):
    from geometry_rl_b200 import _lib, ops
    sm = _lib.sm_count()
    expect = groups * host_slots(b_env * groups, groups, sm) if groups > 1 else max(1, min(b_env, 2 * sm))
    assert ops.critic_partials(b_env * groups, groups) == expect


def test_slots_are_clamped_to_the_graphs_of_a_group():
    assert host_slots(101 * 1, 101, 148) == 1           # Bg = 1
    assert host_slots(17 * 2, 17, 148) == 2             # ceil(296 / 17) = 18 > Bg = 2
    assert host_slots(17 * 4096, 17, 148) == 18
    assert host_slots(101 * 1000, 101, 148) == 3
    assert host_slots(300 * 4, 300, 148) == 1           # more groups than 2 SMs: one slot each


@pytest.fixture(scope="module")
def lib():
    from geometry_rl_b200.csrc import build as b
    b.build()
    from geometry_rl_b200 import _lib
    return _lib


def _desc(lib, **kw):
    fake = 0x1000  # never dereferenced: every case below fails validation before a launch
    base = dict(n_graphs=8, n_tokens=5, n_feat=15, n_partials=4, eps=1e-5, count=8 * 5 * 64.0, x=fake, w1=fake, b1=fake,
                gamma=fake, beta=fake, stats=fake, stat_partials=fake, ysum=fake, grad_ysum=fake, bstats=fake,
                grad_partials=fake, n_groups=1)
    base.update(kw)
    return lib.GrlCriticDesc(**base)


def test_group_arguments_are_checked(lib):
    h = lib.load()
    EINVAL, EUNSUPPORTED = -1, -2
    invalid = [_desc(lib, n_groups=0), _desc(lib, n_groups=-2), _desc(lib, n_groups=3, n_partials=3),  # 8 % 3
               _desc(lib, n_groups=2, n_partials=3),                                                   # 3 % 2
               _desc(lib, n_groups=16, n_partials=16)]                                                 # > n_graphs
    for fn in ("grl_critic_inner_stats", "grl_critic_inner_fwd", "grl_critic_inner_bwd_stats", "grl_critic_inner_bwd"):
        for d in invalid:
            assert getattr(h, fn)(C.byref(d), None) == EINVAL, f"{fn}: {lib.last_error()}"
    for fn in ("grl_critic_inner_bwd_stats", "grl_critic_inner_bwd"):
        for g in (2, 4, 8):
            d = _desc(lib, n_groups=g, n_partials=8)
            assert getattr(h, fn)(C.byref(d), None) == EUNSUPPORTED, f"{fn} n_groups={g}: {lib.last_error()}"
        assert "n_groups" in lib.last_error()


def test_descriptor_keeps_n_groups_last(lib):
    """n_groups is appended: every earlier field keeps its offset."""
    names = [f for f, _ in lib.GrlCriticDesc._fields_]
    assert names[-1] == "n_groups" and names[:-1] == ["n_graphs", "n_tokens", "n_feat", "n_partials", "eps", "count", "x",
                                                        "w1", "b1", "gamma", "beta", "stats", "stat_partials", "ysum",
                                                        "grad_ysum", "bstats", "grad_partials"]
