"""Size-independent properties at BASELINE.json's full size: the 2^20-point C5a contour
grid (Malama partial penetration) that bench.py times.  The oracle needs ~50 ms of CPU
per point, so here it only checks a random sample; the rest are invariants."""
import os

import numpy as np
import pytest

import bench
import unconfined_b200 as ub
from oracle import oracle
from helpers import check_parity, oracle_with_noise

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def c5a():
    ub.force_kernel(None)
    d, t, r, z = bench.c5a_grid(0)
    p, tD, sv, rD, zD, lay = bench.derive(d, t, r, z, ub)
    prm = ub.Params(p)
    s, ds, fl = ub.eval_grid(prm, tD, sv, rD, zD, lay, want_flags=True)
    return dict(p=p, prm=prm, tD=tD, sv=sv, rD=rD, zD=zD, lay=lay, s=s, ds=ds, fl=fl)


def test_full_grid_shape_determinism_and_finiteness(c5a):
    g = c5a
    assert g["s"].shape == (8, 1024, 128) and g["s"].size == 2 ** 20
    s2, ds2 = ub.eval_grid(g["prm"], g["tD"], g["sv"], g["rD"], g["zD"], g["lay"])
    assert np.array_equal(s2, g["s"], equal_nan=True) and np.array_equal(ds2, g["ds"], equal_nan=True)
    clean = g["fl"] == 0
    assert clean.mean() > 0.97
    # non-finite results are data, as in the reference (NaN totlap entries, invlap.f90:71-74)
    assert np.isfinite(g["s"][clean]).mean() > 0.97


def test_full_grid_is_finite_where_the_qd_table_is_ill_conditioned(c5a):
    """At these early-time points (|s| ~ 1e-7) the 128-z kernel's de Hoog, with its reciprocal-based
    q-d division, broke down to NaN where the reference's Smith division stays finite; such an
    inversion is redone with the reference's division.  On this grid every result is finite."""
    g = c5a
    assert np.isfinite(g["s"]).all() and np.isfinite(g["ds"]).all()
    it, ir, iz = np.array([0, 0, 0]), np.array([691, 765, 1023]), np.array([8, 8, 7])
    args = (g["tD"][it], g["sv"][it], g["rD"][ir], g["zD"][iz], g["lay"][iz])
    so, do, _ = oracle.eval_points(oracle.Params(g["p"]), *args)
    assert np.all(np.abs(g["s"][it, ir, iz] - so) < 1e-6 * np.abs(so))
    assert np.all(np.abs(g["ds"][it, ir, iz] - do) < 1e-6 * np.abs(do))


def test_full_grid_sharding_invariance(c5a):
    g = c5a
    half = 512
    sa, da = ub.eval_grid(g["prm"], g["tD"], g["sv"], g["rD"][:half], g["zD"], g["lay"])
    sb, db = ub.eval_grid(g["prm"], g["tD"], g["sv"], g["rD"][half:], g["zD"], g["lay"])
    assert np.array_equal(np.concatenate([sa, sb], axis=1), g["s"], equal_nan=True)
    assert np.array_equal(np.concatenate([da, db], axis=1), g["ds"], equal_nan=True)


def test_full_grid_physics_monotone_in_time_and_radius(c5a):
    g = c5a
    # away from the overflow-affected smallest radii, from the water table (where the
    # reference's double-precision formulas are rounding noise at early time, see
    # malama-partpen in DESIGN.md) and from the earliest times
    s = g["s"][3:, 64:, :100]
    assert np.isfinite(s).all()
    scale = np.abs(s).max()
    assert (np.diff(s, axis=0) > -1e-6 * scale).all()      # drawdown grows with time (step pumping)
    late = g["s"][-1, 64:, 64]
    assert (np.diff(late) < 1e-8 * scale).all()             # and decays with distance


def test_full_grid_random_sample_against_oracle(c5a):
    g = c5a
    rng = np.random.default_rng(7)
    n = 256
    it, ir, iz = rng.integers(0, 8, n), rng.integers(0, 1024, n), rng.integers(0, 128, n)
    args = (g["tD"][it], g["sv"][it], g["rD"][ir], g["zD"][iz], g["lay"][iz])
    po = oracle.Params(g["p"])
    # eight jitter draws: with two, the envelope of the heavy-tailed noise is under-sampled at the
    # ill-conditioned points (the sample's point 179, z = 1 at early time, |s| = 2.6e-9: spread
    # 1.6e-15 from two draws, 8.1e-15 from eight or thirty-two)
    so, do, sps, spd = oracle_with_noise(po, args, points=True, nsamples=8)
    _, _, fo = oracle.eval_points(po, *args)
    assert np.array_equal(fo, g["fl"][it, ir, iz])
    # flagged points included: fresh mode uses infint = 0 on both sides
    well = check_parity(g["s"][it, ir, iz], g["ds"][it, ir, iz], so, do, sps, spd, what="C5a sample")
    print('well-conditioned fraction of the sample:', well)
    assert well > 0.3     # a good share of the sample is well-conditioned and held to 1e-9 outright


def test_grid_kernel_equals_point_kernel_on_sample(c5a):
    g = c5a
    rng = np.random.default_rng(11)
    n = 4096
    it, ir, iz = rng.integers(0, 8, n), rng.integers(64, 1024, n), rng.integers(0, 128, n)
    sp_, dp_ = ub.eval_points(g["prm"], g["tD"][it], g["sv"][it], g["rD"][ir], g["zD"][iz], g["lay"][iz])
    ref = g["s"][it, ir, iz]
    rel = np.abs(sp_ - ref) / np.maximum(np.abs(ref), 1e-300)
    # two different summation orders of the same arithmetic: agree far below the parity bar
    # except where the result itself is rounding noise (tiny early-time drawdowns)
    assert np.median(rel) < 1e-12
    assert (rel < 1e-6).mean() > 0.98


def test_small_radius_columns_overflow_flow_matches_oracle(c5a):
    """The few smallest radii of the C5a grid are where the reference's cosh/sinh overflow:
    Wynn truncation, sentinel and stale flags of the 128-z persistent kernel (which stops
    evaluating a p once every z's series is settled) must match the oracle exactly, and the
    finite results must agree."""
    g = c5a
    ir = np.arange(0, 12)
    it = np.array([1, 6])
    po = oracle.Params(g["p"])
    so, do, fo = oracle.eval_grid(po, g["tD"][it], g["sv"][it], g["rD"][ir], g["zD"], g["lay"], carry=False)
    sg, dg, fg = g["s"][it][:, ir], g["ds"][it][:, ir], g["fl"][it][:, ir]
    assert np.array_equal(fo, fg)
    assert np.array_equal(np.isnan(so), np.isnan(sg))
    # the overflow regime is really exercised: at these radii a/sqrt(kappa) exceeds 710
    assert g["p"]["j0z"][-1] / g["rD"][0] / np.sqrt(g["p"]["kappa"]) > 1000.0
    args = (g["tD"][it], g["sv"][it], g["rD"][ir], g["zD"], g["lay"])
    so2, do2, sps, spd = oracle_with_noise(po, args, nsamples=3)
    check_parity(sg, dg, so2, do2, sps, spd, what="C5a small radii")


def test_small_radius_columns_reference_compatible_mode_with_carry(c5a):
    """The benchmarked kernel in the reference's own mode: stale tanh-sinh abscissae
    (driver.f90:121-126) and the stale-infint carry (driver.f90:205-214) over a sub-grid whose
    smallest radii overflow, preceded and followed by healthy columns, two times.  Every point
    is compared with oracle.eval_grid(carry=True); nothing is masked."""
    g = c5a
    ir = np.array([40, 0, 1, 300, 2, 5, 3])
    it = np.array([1, 6])
    tD, sv, rD = g["tD"][it], g["sv"][it], g["rD"][ir]
    sc = float(g["p"]["j0z"][sv[0] - 1] / rD[0])
    po = oracle.Params(g["p"])
    args = (tD, sv, rD, g["zD"], g["lay"])
    so, do, sps, spd = oracle_with_noise(po, args, ts_scale=sc, carry=True, nsamples=2)
    _, _, fo = oracle.eval_grid(po, *args, ts_scale=sc, carry=True)
    sg, dg, fg = ub.eval_grid(g["prm"], *args, ts_scale=sc, want_flags=True)
    assert np.array_equal(fo, fg)      # (no point of this grid is stale: the carry is exercised on
    check_parity(sg, dg, so, do, sps, spd, what="C5a carry")   # the 128-z kernel in test_gpu_parity.py)


def test_grid8_equals_lanes_z_kernel(c5a):
    """The persistent 128-z kernel and the 64-z lanes<->z kernel implement the same arithmetic
    except for the z-recurrence of the exponentials: results agree far below the parity bar."""
    g = c5a
    ub.force_kernel("grid2")
    try:
        s2, d2, f2 = ub.eval_grid(g["prm"], g["tD"][2:4], g["sv"][2:4], g["rD"][::16], g["zD"], g["lay"], want_flags=True)
    finally:
        ub.force_kernel(None)
    s4, f4 = g["s"][2:4][:, ::16], g["fl"][2:4][:, ::16]
    assert np.array_equal(f2, f4)
    ok = np.isfinite(s2) & np.isfinite(s4)
    rel = np.abs(s4[ok] - s2[ok]) / np.maximum(np.abs(s2[ok]), 1e-300)
    assert np.median(rel) < 1e-12 and (rel < 1e-7).mean() > 0.98


def test_grid8_on_odd_column_counts_and_ragged_z(c5a):
    """lh_grid8_kernel (8 z-slots per lane, two Laplace parameters per warp) against the
    lanes<->z kernel on shapes that exercise its edges: odd numbers of columns, z-blocks that
    are not full, a second partial z-block."""
    g = c5a
    for nr, nt, zsel in ((5, 1, slice(0, 128)), (3, 3, slice(0, 100)), (2, 1, slice(0, 128, 1))):
        tD, sv = g["tD"][2:2 + nt], g["sv"][2:2 + nt]
        rD = g["rD"][100:100 + 37 * nr:37]
        zD, lay = g["zD"][zsel], g["lay"][zsel]
        s8, d8, f8 = ub.eval_grid(g["prm"], tD, sv, rD, zD, lay, want_flags=True)
        ub.force_kernel("grid2")
        try:
            s4, d4, f4 = ub.eval_grid(g["prm"], tD, sv, rD, zD, lay, want_flags=True)
        finally:
            ub.force_kernel(None)
        assert np.array_equal(f8, f4)
        assert np.array_equal(np.isnan(s8), np.isnan(s4))
        ok = np.isfinite(s4)
        rel = np.abs(s8[ok] - s4[ok]) / np.maximum(np.abs(s4[ok]), 1e-300)
        assert np.median(rel) < 1e-12 and (rel < 1e-7).mean() > 0.98, (nr, nt, np.median(rel))
    # 200 z = one full and one partial z-block, equally spaced; against the point kernel
    z = np.linspace(0.0, 1.0, 200)
    lay = ub.zlay(z, g["p"]["lD"], g["p"]["dD"])
    tD, sv, rD = g["tD"][4:5], g["sv"][4:5], g["rD"][300:303]
    s8, d8 = ub.eval_grid(g["prm"], tD, sv, rD, z, lay)
    ub.force_kernel("point")
    try:
        sp_, dp_ = ub.eval_grid(g["prm"], tD, sv, rD, z, lay)
    finally:
        ub.force_kernel(None)
    ok = np.isfinite(sp_)
    rel = np.abs(s8[ok] - sp_[ok]) / np.maximum(np.abs(sp_[ok]), 1e-300)
    assert np.median(rel) < 1e-12 and (rel < 1e-6).mean() > 0.98


def test_single_process_multi_gpu_sharding_is_bitwise_invariant(c5a):
    """unc_eval_grid_ex(ngpu = all) on one grid, columns split across the visible GPUs (shard
    boundaries fall inside time rows when nt is not a multiple of ngpu), with and without the
    carry: bitwise the single-GPU result.  With one visible GPU this degenerates to ngpu=1."""
    g = c5a
    n = ub.device_count()
    tD, sv, rD = g["tD"][1:4], g["sv"][1:4], g["rD"][:90]
    s1, d1, f1 = ub.eval_grid(g["prm"], tD, sv, rD, g["zD"], g["lay"], ngpu=1, want_flags=True)
    assert np.array_equal(s1, g["s"][1:4][:, :90], equal_nan=True)
    for k in sorted({n, max(1, n - 1)}):
        sk, dk, fk = ub.eval_grid(g["prm"], tD, sv, rD, g["zD"], g["lay"], ngpu=k, want_flags=True)
        assert np.array_equal(sk, s1, equal_nan=True) and np.array_equal(dk, d1, equal_nan=True)
        assert np.array_equal(fk, f1)
    sc = float(g["p"]["j0z"][sv[0] - 1] / rD[40])
    a1 = ub.eval_grid(g["prm"], tD, sv, rD, g["zD"], g["lay"], ts_scale=sc, ngpu=1)
    an = ub.eval_grid(g["prm"], tD, sv, rD, g["zD"], g["lay"], ts_scale=sc, ngpu=0)
    assert np.array_equal(a1[0], an[0], equal_nan=True) and np.array_equal(a1[1], an[1], equal_nan=True)
