"""Every row-solver layout of ALS-WRMF (als.cu: als_layout picks C CTAs per row and kTile staged
neighbour rows per step from k and the device's shared memory) against the float64 normal equations
of oracle/als_systems.py, one half-pass at a time: the user pass against the initial item factors,
the item pass against the user factors the device computed.  Every solved row's backward error must
stay under 8 (k + deg + n_fixed) eps, its forward error under that times cond(M) where cond(M) <= 1e8;
rows without neighbours must be exactly zero and inactive rows untouched.

The sweep runs k values at every layout boundary and at the residues mod 8, 32 and 64 that the
kernels' pitches and tiles depend on, with rows whose degree is 0, 1, kTile - 1, kTile, kTile + 1,
2 kTile and 2 kTile + 1.  The last test asserts that every layout of the device ran at least twice
and prints, per layout, the k values run, the largest backward error and where it occurred."""
import collections

import numpy as np
import pytest

from oracle import als_systems as A

pytestmark = pytest.mark.gpu

B200_SMEM = (228 * 1024, 227 * 1024)   # shared memory per SM, opt-in per block


def _device_smem():
    """The device's shared memory sizes; the B200's where no device is visible (collection on a CPU box)."""
    import torch
    if not torch.cuda.is_available():
        return B200_SMEM
    p = torch.cuda.get_device_properties(torch.cuda.current_device())
    return p.shared_memory_per_multiprocessor, p.shared_memory_per_block_optin


# The cluster kernel's static shared memory (0 or 1 KB) moves two boundaries by one.  A k is credited
# to a layout only where both give the same one.
_SMEM = _device_smem()
_TABLES = [A.layout_table(*_SMEM, cluster_static_smem=s) for s in (0, 1024)]


def _layout(k):
    a, b = (A.als_layout(k, *_SMEM, cluster_static_smem=s) for s in (0, 1024))
    return a if a == b else None


K_SWEEP = sorted({1, 2, 3, 5, 8, 9, 16, 17, 31, 32, 33, 63, 65, 69, 70, 72, 76, 77, 96, 127, 128, 129, 164,
                  165, 166, 191, 192, 193, 198, 199, 216, 220, 226, 227, 232, 240, 243, 255, 256}
                 | {k for t in _TABLES for _c, _t, a, b in t for k in (a, b)})
K_INTERIOR = [20, 72, 120, 180, 205, 220, 232, 250]   # one per layout of the B200

# (C, kTile) -> [(k, largest eta, largest eta / bound, where the largest eta was)], one entry per
# checked run; the k values swept
_RUNS = collections.defaultdict(list)
_SWEPT = set()


def _device():
    import torch
    return torch.cuda.current_device()


def _edges(k):
    """Degrees at the staging-step edges of k's kTile (of both candidates where k is ambiguous)."""
    tiles = {A.als_layout(k, *_SMEM, cluster_static_smem=s)[1] for s in (0, 1024)}
    return sorted({d for t in tiles for d in (0, 1, t - 1, t, t + 1, 2 * t, 2 * t + 1)})


def _train(p, k, epochs, c_pos, reg, u=None, v=None):
    from mfrec_b200 import _native
    u = (p["u0"] if u is None else u).copy()
    v = (p["v0"] if v is None else v).copy()
    _native.train_als_wrmf(epochs, k, u, v, p["ur"], p["uc"], p["ir"], p["ic"], p["nu"], p["ni"], c_pos, reg,
                           ctx=_native.default_context(_device()))
    return u, v


def _check_one_epoch(p, k, what, c_pos=1, reg=0.015):
    """One epoch on the device, both half-passes checked, the run recorded under ``what``."""
    u1, v1 = _train(p, k, 1, c_pos, reg)
    runs = []
    for side, d in (("users", A.check_half_pass(p["u0"], p["v0"], v1, p["ur"], p["uc"], c_pos, reg, p["nu"])),
                    ("items", A.check_half_pass(v1, p["u0"], u1, p["ir"], p["ic"], c_pos, reg, p["ni"]))):
        i = int(np.argmax(d["eta"]))
        runs.append((d["eta"][i], (d["eta"] / d["bound"]).max(),
                     "%s k=%d %s row %d deg %d cond %.1e" % (what, k, side, d["row"][i], d["deg"][i], d["cond"][i])))
    lay = _layout(k)
    if lay is not None:
        eta, _, where = max(runs)
        _RUNS[lay].append((k, eta, max(r[1] for r in runs), where))


@pytest.mark.parametrize("k", K_SWEEP)
def test_sweep_every_layout(k):
    p = A.implicit_problem(k, 300, 200, 4000, seed=k, degrees=_edges(k), hot=60)
    _check_one_epoch(p, k, "sweep")
    _SWEPT.add(k)


@pytest.mark.parametrize("c_pos,reg", [(0, 1e-6), (0, 3.0), (40, 1e-6), (40, 3.0)])
@pytest.mark.parametrize("k", K_INTERIOR)
def test_non_default_parameters(k, c_pos, reg):
    """c_pos and reg other than the reference's 1 and 0.015, and a user and an item that list one
    neighbour twice."""
    p = A.implicit_problem(k, 150, 100, 1800, seed=k + c_pos, degrees=_edges(k), hot=30, duplicate=True)
    _check_one_epoch(p, k, "c_pos=%d reg=%g" % (c_pos, reg), c_pos, reg)


@pytest.mark.parametrize("c_pos,reg", [(1, 0.015), (40, 1e-6)])
def test_fewer_fixed_rows_than_k(c_pos, reg):
    """k = 232 with 150 items and 200 users: HH is singular on both sides, reg alone keeps M definite."""
    k = 232
    p = A.implicit_problem(k, 200, 150, 2500, seed=3, degrees=_edges(k), hot=40, duplicate=True)
    _check_one_epoch(p, k, "fewer fixed rows, c_pos=%d reg=%g" % (c_pos, reg), c_pos, reg)


@pytest.mark.parametrize("k", [72, 120, 220, 232])
def test_hot_row(k):
    """Item 0 with more than 1,500 neighbours: many staging steps, the last one partial or full."""
    p = A.implicit_problem(k, 1650, 200, 3000, seed=k, degrees=_edges(k), hot=1550)
    assert p["ir"][1] > 1500
    _check_one_epoch(p, k, "hot row")


@pytest.mark.parametrize("k", [72, 220, 232])
def test_two_epochs_match_c_oracle(k):
    """The three layouts no earlier test ran -- (1, 16), (2, 8), (3, 32) on a B200 -- against the C
    oracle over two epochs, at the standard of tests/test_als_large_k_gpu.py."""
    from oracle import cpu
    p = A.implicit_problem(k, 300, 200, 4000, seed=k + 1, degrees=_edges(k), hot=60, duplicate=True)
    u0, v0 = p["u0"].copy(), p["v0"].copy()
    cpu.als_wrmf(2, k, u0, v0, p["ur"], p["uc"], p["ir"], p["ic"], 1, 0.015)
    u1, v1 = _train(p, k, 2, 1, 0.015)
    np.testing.assert_allclose(u1, u0, rtol=1e-8, atol=1e-11)
    np.testing.assert_allclose(v1, v0, rtol=1e-8, atol=1e-11)


@pytest.mark.parametrize("k", K_INTERIOR)
def test_deterministic(k):
    p = A.implicit_problem(k, 300, 200, 4000, seed=k + 2, degrees=_edges(k), hot=60, duplicate=True)
    a, b = _train(p, k, 2, 1, 0.015), _train(p, k, 2, 1, 0.015)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("k", [72, 220, 232])
def test_three_shards_on_one_device_bit_identical(k):
    """Three shards on one device, each solution stored into three copies, in the layouts no earlier
    test ran, against the one-device call (one shard, one copy)."""
    from mfrec_b200 import _native
    d = _device()
    p = A.implicit_problem(k, 300, 200, 4000, seed=k + 3, degrees=_edges(k), hot=60, duplicate=True)
    u0, v0 = _train(p, k, 2, 1, 0.015)
    u1, v1 = p["u0"].copy(), p["v0"].copy()
    _native.train_als_wrmf_multi([d] * 3, 2, k, u1, v1, p["ur"], p["uc"], p["ir"], p["ic"], p["nu"], p["ni"], 1, 0.015)
    assert np.isfinite(u0).all() and np.isfinite(v0).all()
    assert np.array_equal(u1, u0) and np.array_equal(v1, v0)


def test_every_layout_ran_twice():
    """Runs last: every (C, kTile) of this device's table ran at least twice in this session."""
    if not _SWEPT:
        pytest.skip("the sweep did not run in this session")
    lines = ["device shared memory: %d B per SM, %d B opt-in per block" % _SMEM,
             "%-9s %-20s %-56s %-11s %-11s %s" % ("(C, kT)", "k range", "k run", "max eta", "eta/bound",
                                                  "largest eta at")]
    missing = []
    for c, t, a, b in _TABLES[0]:
        runs = _RUNS.get((c, t), [])
        ks = sorted({r[0] for r in runs})
        other = [(s[2], s[3]) for s in _TABLES[1] if s[:2] == (c, t)]
        rng = "%d..%d" % (a, b) + ("" if other == [(a, b)] else " (%d..%d)" % other[0])
        top = max(runs, key=lambda r: r[1], default=(0, float("nan"), float("nan"), "-"))
        ratio = max((r[2] for r in runs), default=float("nan"))
        lines.append("%-9s %-20s %-56s %-11.2e %-11.2e %s" % ("(%d, %d)" % (c, t), rng, ",".join(map(str, ks)),
                                                            top[1], ratio, top[3]))
        if len(ks) < 2:
            missing.append((c, t))
    print("\n" + "\n".join(lines))
    assert not missing, "layouts run fewer than twice: %s" % missing
