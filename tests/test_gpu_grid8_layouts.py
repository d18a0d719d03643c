"""lh_grid8_kernel (grid8.cuh) against the oracle point by point on every z-layout path it takes.

Per item (one (t,r) column x up to 128 z: lanes hl = 0..15, slots k = 0..7, z index hl + 16 k) the
kernel picks its code from the z-list and zLay alone: the equally-spaced check, the common layer
Lc, the one exception slot kx whose off-layer lanes lie on one other layer Lb, K0Z (k0 of Lc is
zero), the padding slots, and slow8_run for everything else.  `classify` below restates those
decisions; the designed z-lists are built from each deck's lD, dD so that every (kx, K0Z) pair and
Lb on both sides of Lc runs on the hot path, and every slow-path reason is taken.  The statistical
tests of test_gpu_parity.py / test_gpu_fullsize.py allow a few per cent of a grid to miss; here no
point is excused: the oracle at every z of the exception slot, on both sides of each boundary and
at the ends of every other slot, and the hot path against the exact path at all 128 z.

Reachability with geometric zLay (oracle.zlay): layers are monotone in z, so on an equally spaced
list a boundary inside slot kx leaves every later slot off Lc as well, unless slot kx is the
item's last slot.  Hence kx = 0 cannot be reached (slot 1 would be off too, and an item of at most
16 z is never equally spaced), kx = 1 only by the 17..32-z tail of a column longer than 128 z,
and kx < 7 of a descending list not at all (its padding slots take the lowest layer present,
which is Lb, so they are off as well): descending lists reach kx = 7 only."""
import numpy as np
import pytest

import unconfined_b200 as ub
from oracle import oracle
from helpers import load_deck, check_parity, oracle_with_noise, RTOL, NOISE_K

EPS = 2.220446049250313e-16
ZB, GL, ZL = 128, 16, 8
K0_MODELS = (1, 2, 3, 5)      # k0 is zero outside the screen (layer 2) of these models
DECKS = {0: "theis-input.dat", 1: "hantush-input.dat", 2: "hantush-storage-input.dat", 3: "cape-cod-moench.in",
         4: "malama-fullpen-input.dat", 5: "malama-partpen-input.dat", 6: "mishra-neuman-malama.in"}
NEUMAN74 = "cape-cod-neuman74.in"


# ------------------------------------------------------------------------------------------------
# item classifier: grid8.cuh:100-123 (descriptor, T-job) and :304-347 (p-job), one block of <= 128 z
# ------------------------------------------------------------------------------------------------
def classify(zD, zLay, model):
    """Layers are 1-based here (as in zLay); the kernel's Lc, Lb, Lx are 0-based."""
    z = np.asarray(zD, np.float64)
    lay = np.asarray(zLay, np.int64)
    nzv = len(z)
    assert 1 <= nzv <= ZB
    idx = np.arange(GL)[:, None] + GL * np.arange(ZL)[None, :]            # [hl, k] -> hl + 16 k
    valid = idx < nzv                                                      # zvalid (:101-106)
    zz = np.where(valid, z[np.minimum(idx, nzv - 1)], 0.0)
    ll = np.where(valid, lay[np.minimum(idx, nzv - 1)], 0)
    mm = 0                                                                 # lay_mask, za (:107-115)
    za = np.float32(0.0)
    for zi, li in zip(z, lay):
        mm |= 1 << int(li - 1)
        za = max(za, np.float32(np.float32(abs(zi)) * np.float32(1.0000002)))
    D = zz[0, 1] - zz[0, 0]                                                # lane 0, slots 0 and 1 (:117)
    tol = 4.0 * EPS * float(za)                                            # :118
    dev = 0.0
    uni = bool(valid[0, 0] and valid[0, 1])                                # :119-123
    for k in range(ZL - 1):
        both = valid[:, k] & valid[:, k + 1]
        d = np.abs((zz[:, k + 1] - zz[:, k]) - D)[both]
        if len(d):
            dev = max(dev, float(d.max()))
            if not np.all(d <= tol):
                uni = False
    L0 = (mm & -mm).bit_length()                                           # lowest layer present (:297)
    myL = np.where(valid, ll, L0)                                          # padding slots (:314)
    Lc = int(myL[0, 0])                                                    # :327
    off = [k for k in range(ZL) if not np.all(myL[:, k] == Lc)]            # offmask (:328-331)
    kx = off[0] if len(off) == 1 else -1                                   # :332
    hot_ok = len(off) <= 1                                                 # :333
    Lb = Lc
    if kx >= 0:
        Lx = np.where(valid[:, kx], myL[:, kx], Lc)                        # :334-341
        offl = np.nonzero(Lx != Lc)[0]
        if len(offl):
            Lb = int(Lx[offl[0]])                                          # :342-343
        if not np.all((Lx == Lc) | (Lx == Lb)):
            hot_ok = False                                                 # :344
    k0z = model in K0_MODELS and Lc != 2                                   # :347 (0-based Lc != 1)
    if nzv <= GL:
        reason = "tail of 16 z or fewer"
    elif not uni:
        reason = "not equally spaced"
    elif len(off) > 1:
        reason = "several slots off the common layer"
    elif not hot_ok:
        reason = "exception slot on two other layers"
    else:
        reason = None
    return dict(zuni=uni, offmask=sum(1 << k for k in off), kx=kx, Lc=Lc, Lb=Lb, K0Z=k0z, hot_ok=hot_ok,
                reason=reason, tol=tol, dev=dev, D=D, nzv=nzv)


def blocks(nz):
    return [(b, min(ZB, nz - b)) for b in range(0, nz, ZB)]


def hot_key(c):
    """(kx, K0Z, direction of Lb) of a hot-path item; direction 0 when no lane is off Lc."""
    return (c["kx"], c["K0Z"], int(np.sign(c["Lb"] - c["Lc"])))


# ------------------------------------------------------------------------------------------------
# classifier self-check on hand-worked blocks (no GPU)
# ------------------------------------------------------------------------------------------------
def test_classifier_hand_worked_blocks():
    z = np.linspace(0.1, 0.6, 128)
    c = classify(z, np.ones(128, int), 1)           # one layer: hot, no exception slot, k0 of layer 1 is zero
    assert (c["zuni"], c["kx"], c["Lc"], c["K0Z"], c["reason"]) == (True, -1, 1, True, None)
    assert classify(z, np.ones(128, int), 0)["K0Z"] is False      # Theis: k0 is not zero
    lay = np.where(np.arange(128) < 115, 1, 2)     # boundary between lanes 2 and 3 of slot 7
    c = classify(z, lay, 3)
    assert (c["kx"], c["Lc"], c["Lb"], c["K0Z"], c["offmask"], c["reason"]) == (7, 1, 2, True, 0x80, None)
    c = classify(z, np.where(np.arange(128) < 100, 2, 3), 3)     # boundary in slot 6: slots 6 and 7 off
    assert (c["offmask"], c["kx"], c["K0Z"], c["reason"]) == (0xC0, -1, False, "several slots off the common layer")
    c = classify(z[:40], np.where(np.arange(40) < 36, 1, 2), 5)   # 40 z: lanes 8..15 of slot 2 pad
    assert (c["kx"], c["Lb"], c["offmask"], c["reason"]) == (2, 2, 0x04, None)
    zd = z[::-1][:120]                               # descending, 120 z: Lc = 3 on top, Lb = 2 below
    c = classify(zd, np.where(np.arange(120) < 115, 3, 2), 1)
    assert (c["Lc"], c["kx"], c["Lb"], c["K0Z"], c["reason"]) == (3, 7, 2, True, None)
    c = classify(zd[:100], np.where(np.arange(100) < 97, 3, 2), 1)   # ... 100 z: padding slot 7 takes L0 = 2
    assert c["offmask"] == 0xC0 and c["reason"] == "several slots off the common layer"
    lay = np.where(np.arange(128) < 118, 1, np.where(np.arange(128) < 124, 2, 3))
    assert classify(z, lay, 1)["reason"] == "exception slot on two other layers"
    assert classify(z[:16], np.ones(16, int), 1)["reason"] == "tail of 16 z or fewer"
    assert classify(np.full(64, 0.3), np.ones(64, int), 1)["reason"] is None      # D = 0 is equally spaced
    # tolerance: 4 ulp of max|z| (as float, times 1.0000002); deviations measured on exact dyadic z
    for c_ulp, ok in ((3.9, True), (5.0, False)):
        zt, _ = tolerance_list(c_ulp)
        c = classify(zt, np.ones(128, int), 1)
        assert c["zuni"] is ok and abs(c["dev"] / (c["tol"] / 4) - c_ulp) < 0.15, (c_ulp, c["dev"] / (c["tol"] / 4))


def tolerance_list(c_ulp):
    """128 dyadic z, 0.40625 + i/256 (up to 0.90234375): every z and every step below is exact.
    Lane 0 keeps the exact spacing (it defines D); every other lane's slot k moves up by k*n
    doubles of [0.5, 1), n chosen so that each of those lanes' slot-to-slot steps deviates from D
    by about c ulp of max|z|, all with the same sign (7 c ulp of drift by slot 7)."""
    i = np.arange(128)
    z = 0.40625 + i / 256.0
    za = float(np.float32(np.float32(z.max()) * np.float32(1.0000002)))
    s = 2.0 ** -53                                   # spacing of the doubles in [0.5, 1)
    n = int(round(c_ulp * EPS * za / s))
    zt = z + np.where(i % GL != 0, (i // GL) * n * s, 0.0)
    return zt, n * s / (EPS * za)


# ------------------------------------------------------------------------------------------------
# designed z-lists
# ------------------------------------------------------------------------------------------------
_DECK_CACHE = {}


def deck_of(name):
    if name not in _DECK_CACHE:
        d, pd = load_deck(name)
        tD = np.array([d["tD"][len(d["tD"]) // 3], d["tD"][(3 * len(d["tD"])) // 4]]) if len(d["tD"]) > 1 \
            else np.array([d["tD"][0], 30.0 * d["tD"][0]])
        pq = dict(pd, j0z=oracle.j0_zeros(max(d["j0s"]) + pd["gl_nacc"] + 1))
        _DECK_CACHE[name] = (d, pq, tD, oracle.split_index(tD, d["j0s"]))
    return _DECK_CACHE[name]


def layer_range(pq, L):
    lD1, dD1 = 1.0 - pq["lD"], 1.0 - pq["dD"]
    return {1: (0.0, lD1), 2: (lD1, dD1), 3: (dD1, 1.0)}[L]


def boundary_list(pq, Lc, Lb, g, nz, at=False):
    """Equally spaced list of nz z: index < g on layer Lc, index >= g on layer Lb (|Lc - Lb| = 1),
    the boundary halfway between z[g-1] and z[g] (at=True: the one of the two on the upper layer
    exactly on it).  Ascending when Lb is above Lc, descending otherwise; the list keeps clear of
    the other layers and of z = 1 (which geometric zLay puts on layer 2)."""
    up = Lb > Lc
    B = layer_range(pq, max(Lc, Lb))[0]
    lo_c, hi_c = layer_range(pq, Lc)
    lo_b, hi_b = layer_range(pq, Lb)
    room_c = (B - lo_c) if up else (hi_c - B)
    room_b = (hi_b - B) if up else (B - lo_b)
    h = 0.9 * min(room_c / (g + 0.5), room_b / (nz - g + 1.5))
    i = np.arange(nz)
    if up:
        z = B + (i - g + (0.0 if at else 0.5)) * h
    else:
        z = B - (i - g + (1.0 if at else 0.5)) * h
    lay = oracle.zlay(z, pq["lD"], pq["dD"])
    assert np.array_equal(lay, np.where(i < g, Lc, Lb)), (Lc, Lb, g, nz, lay)
    return z, lay


class Case:
    def __init__(self, name, deck, z, lay, rD=(0.6, 1.8), nudge=True):
        self.name, self.deck, self.z, self.lay, self.rD, self.nudge = name, deck, np.asarray(z), np.asarray(lay), rD, nudge
        _, pq, _, _ = deck_of(deck)
        self.model = pq["model"]
        self.layers = (pq["lD"], pq["dD"])
        self.cls = [classify(self.z[b:b + n], self.lay[b:b + n], self.model) for b, n in blocks(len(self.z))]

    def __repr__(self):
        return self.name


JS = (0, 1, 8, 15)


def exception_case(deck, kx, j, Lc, Lb, at=False):
    """Item whose last slot is kx, boundary between lanes j-1 and j of slot kx (j = 0: between slot
    kx-1 and slot kx).  kx = 1 is the tail of a 128 + 17..32-z column.  A partly filled last slot
    (padding lanes) where j allows it."""
    d, pq, _, _ = deck_of(deck)
    n = 16 if j == 15 else 12 + (kx % 3)
    b0 = ZB if kx == 1 else 0
    if Lb < Lc:                  # descending: full blocks only
        assert kx == 7
        n = 16
    nz = b0 + GL * kx + n
    g = b0 + GL * kx + j
    z, lay = boundary_list(pq, Lc, Lb, g, nz, at=at)
    return Case(f"{deck}:kx{kx}:j{j}:L{Lc}->{Lb}{':at' if at else ''}:nz{nz}", deck, z, lay)


def designed_cases():
    cases = []
    # ascending from layer 1: K0Z for models 1, 2, 3, 5; not for 0, 4
    for m in (0, 1, 2, 3, 4, 5):
        for kx in range(1, 8):
            if (kx + m) % 2 and m in (0, 2, 4, 5) and kx != 7:
                continue
            cases.append(exception_case(DECKS[m], kx, JS[(kx + m) % 4], 1, 2, at=(kx == 3)))
    # ascending from layer 2 (Lb = 3 above): K0Z false for the Hantush-type models
    for deck, kxs in ((DECKS[1], (2, 5)), (DECKS[3], (1, 3, 4, 6, 7)), (NEUMAN74, (2, 5, 7)), (DECKS[5], (4,))):
        for kx in kxs:
            cases.append(exception_case(deck, kx, JS[kx % 4], 2, 3))
    # descending full blocks (Lc on top, Lb below)
    for deck, Lc, j in ((DECKS[1], 3, 8), (DECKS[3], 3, 1), (NEUMAN74, 3, 0), (DECKS[5], 3, 15),
                        (DECKS[2], 2, 8), (DECKS[3], 2, 15), (DECKS[4], 2, 1), (DECKS[6], 2, 15)):
        if deck == DECKS[6]:     # lD = 1: only z = 0 is on layer 1
            z = np.linspace(0.9, 0.0, 128)
            cases.append(Case(f"{deck}:kx7:desc-to-z0", deck, z, oracle.zlay(z, 1.0, 0.0)))
            continue
        cases.append(exception_case(deck, 7, j, Lc, Lc - 1, at=(j == 8)))
    # no exception slot: one layer
    for m, L in ((1, 1), (3, 1), (0, 2), (4, 1), (6, 2)):
        _, pq, _, _ = deck_of(DECKS[m])
        lo, hi = layer_range(pq, L)
        z = np.linspace(lo + 0.05 * (hi - lo), hi - 0.05 * (hi - lo), 96)
        cases.append(Case(f"{DECKS[m]}:one-layer-{L}", DECKS[m], z, oracle.zlay(z, pq["lD"], pq["dD"])))
    return cases


def edge_cases():
    cases = []
    _, pq, _, _ = deck_of(DECKS[1])          # hantush: layer 2 is 0.01 wide
    # two boundaries in one slot: lanes of slot 7 on layers 1, 2 and 3 (slow path)
    B1, B2 = 1 - pq["lD"], 1 - pq["dD"]
    h = (B2 - B1) / 5.5
    z = B1 + (np.arange(128) - 115 + 0.5) * h
    cases.append(Case("hantush:two-boundaries-in-slot-7", DECKS[1], z, oracle.zlay(z, pq["lD"], pq["dD"])))
    # a boundary in slot 3 of a full block: slots 3..7 off (slow path)
    _, pq3, _, _ = deck_of(DECKS[3])
    z, lay = boundary_list(pq3, 1, 2, 3 * GL + 5, 128)
    cases.append(Case("moench:boundary-in-slot-3-of-128", DECKS[3], z, lay))
    # tolerance edge: 3.9 ulp accepted (hot, z advanced from z_first + k D, 27 ulp of drift), 5 rejected
    for c_ulp in (3.9, 5.0):
        z, _ = tolerance_list(c_ulp)
        cases.append(Case(f"hantush:tolerance-{c_ulp}ulp", DECKS[1], z, oracle.zlay(z, pq["lD"], pq["dD"]), nudge=False))
    # all-equal z (D = 0), on layer 1 and exactly on 1 - lD (layer 2)
    for zz in (0.3, B1):
        z = np.full(48, zz)
        cases.append(Case(f"moench:all-equal-{zz:.4f}", DECKS[3], z, oracle.zlay(z, pq3["lD"], pq3["dD"]), nudge=False))
    # z at 0, at 1 - lD, at 1 - dD and at 1, inside a list of 40
    z = np.concatenate([[0.0, 1 - pq3["lD"], 1 - pq3["dD"], 1.0], np.linspace(0.05, 0.95, 36)])
    cases.append(Case("moench:z-at-0-boundaries-1", DECKS[3], z, oracle.zlay(z, pq3["lD"], pq3["dD"])))
    # shuffled list over all three layers: every slot takes its own layers (slow path)
    z = np.random.default_rng(7).permutation(np.linspace(0.0, 0.99, 128))
    cases.append(Case("neuman74:shuffled", NEUMAN74, z, oracle.zlay(z, *[deck_of(NEUMAN74)[1][k] for k in ("lD", "dD")])))
    # multi-block columns, ascending and descending, over all layers
    for i, nz in enumerate((129, 143, 144, 145, 160, 161, 256, 257, 300)):
        deck = (DECKS[1], DECKS[3], DECKS[2], NEUMAN74, DECKS[0])[i % 5]
        _, pqd, _, _ = deck_of(deck)
        for desc in (False, True):
            z = np.linspace(0.02, 0.995, nz)
            if desc:
                z = z[::-1].copy()
            cases.append(Case(f"{deck}:nz{nz}:{'desc' if desc else 'asc'}", deck, z,
                              oracle.zlay(z, pqd["lD"], pqd["dD"]), rD=(0.9,)))
    return cases


def oracle_sample(case):
    """z of each block sampled for the oracle: every z of the exception slot, both sides of every
    layer change, first and last z of every slot."""
    nz = len(case.z)
    sel = set()
    for (b, n), c in zip(blocks(nz), case.cls):
        for k in range(ZL):
            lo, hi = b + GL * k, min(b + GL * k + GL, b + n)
            if lo >= b + n:
                break
            if k == c["kx"]:
                sel.update(range(lo, hi))
            sel.update((lo, hi - 1))
    ch = np.nonzero(np.diff(case.lay) != 0)[0]
    sel.update(ch.tolist())
    sel.update((ch + 1).tolist())
    return np.array(sorted(sel))


def nudged(case):
    """The same list with one z per equally spaced block moved by 16 ulp of max|z|, inside its layer
    and not the largest |z|: lay_mask, za and so eta_max stay the same, the block takes slow8_run.
    (A block of 17..31 z whose lanes 1.. have one slot each has no such z.)  Returns (z, nudged
    indices) or None."""
    z = case.z.copy()
    moved = []
    for (b, n), c in zip(blocks(len(z)), case.cls):
        if c["reason"] is not None or n <= GL:
            continue
        zmax = np.abs(z[b:b + n]).max()
        for i in [b + q for q in (2, 3, 5, 7, 9, 11, 13) if q < n]:
            for sgn in (1.0, -1.0):
                zi = z[i] + sgn * 16 * EPS * zmax
                if not (0.0 <= zi <= 1.0) or abs(zi) >= zmax or abs(z[i]) >= zmax:
                    continue
                if oracle.zlay(np.array([zi]), *case.layers)[0] != case.lay[i]:
                    continue
                trial = z.copy()
                trial[i] = zi
                if classify(trial[b:b + n], case.lay[b:b + n], case.model)["reason"] == "not equally spaced":
                    z = trial
                    moved.append(i)
                    break
            if moved and moved[-1] == i:
                break
    return (z, moved) if moved else None


# ------------------------------------------------------------------------------------------------
# GPU runs
# ------------------------------------------------------------------------------------------------
@pytest.fixture
def gpu():
    assert ub.device_count() >= 1, "no CUDA device: the product path has no CPU fallback"
    ub.force_kernel(None)
    ub.set_carry(True)
    yield
    ub.force_kernel(None)
    ub.set_carry(True)


PAIRS = ((0, 0), (1, -1))      # (mid time, first radius), (late time, last radius)


def grid8_eval(prm, tD, sv, rD, zD, zLay, **kw):
    """ub.eval_grid on lh_grid8_kernel whatever the grid's size: left to itself, the library gives
    small grids (nz < 64 with fewer column CTAs than SMs) to the point kernel.  The forced choice
    takes the 128-z kernel for every nz >= 32 (capi.cu launch_grid), which is asserted here, so
    that every result this file compares, and every item it counts as covered, comes from it."""
    assert len(zD) >= 32, f"nz = {len(zD)} would not run on lh_grid8_kernel"
    ub.force_kernel("grid8")
    try:
        return ub.eval_grid(prm, tD, sv, rD, zD, zLay, want_flags=True, **kw)
    finally:
        ub.force_kernel(None)


def run_case(case):
    """Fresh abscissae (no carry): the kernel on every z of two columns, (mid time, first radius)
    and (late time, last radius); the oracle on the sampled z.  Returns the kernel's (s, ds, flags)
    as [column, z], the sample, the oracle's |value| and noise part of the parity bar
    (NOISE_K * spread) at the sampled points (NaN elsewhere), and the well-conditioned fraction."""
    d, pq, tD, sv = deck_of(case.deck)
    rD = np.asarray(case.rD, float)
    sel = oracle_sample(case)
    out = [np.empty((2, len(case.z))) for _ in range(2)] + [np.empty((2, len(case.z)), np.int32)]
    bars = [np.full(out[0].shape, np.nan) for _ in range(4)]     # |s|, noise of s, |ds|, noise of ds
    wells = []
    for c, (i, k) in enumerate(PAIRS):
        col = (tD[i:i + 1], sv[i:i + 1], rD[k:] if k < 0 else rD[k:k + 1])
        sg, dg, fg = grid8_eval(ub.Params(pq), *col, case.z, case.lay)
        for o, r in zip(out, (sg, dg, fg)):
            o[c] = r[0, 0]
        args = col + (case.z[sel], case.lay[sel])
        so, do, sps, spd = oracle_with_noise(oracle.Params(pq), args, nsamples=3)
        _, _, fo = oracle.eval_grid(oracle.Params(pq), *args, carry=False)
        assert np.array_equal(fo[0, 0], fg[0, 0, sel]), f"{case}: flags differ from the oracle's"
        wells.append(check_parity(sg[:, :, sel], dg[:, :, sel], so, do, sps, spd, what=f"{case} (t{i}, r{k})"))
        bars[0][c, sel], bars[1][c, sel] = np.abs(so[0, 0]), NOISE_K * sps[0, 0]
        bars[2][c, sel], bars[3][c, sel] = np.abs(do[0, 0]), NOISE_K * spd[0, 0]
    return tuple(out), sel, bars, float(np.mean(wells))


def hot_vs_exact(case, res, sel, bars):
    """Every shared z of the equally spaced run (hot path) against the run with one z per block
    nudged (slow8_run): same abscissae, same summation order, only the integrand's rounding
    differs.  Bar at a sampled z: the oracle's parity bar there.  Elsewhere 1e-9 relative; a z
    that misses it gets the oracle's parity bar of its own (the oracle and its noise envelope
    evaluated at that z), never one borrowed from other z."""
    nd = nudged(case)
    if nd is None:
        return 0, 0
    z2, moved = nd
    d, pq, tD, sv = deck_of(case.deck)
    rD = np.asarray(case.rD, float)
    keep = np.ones(len(case.z), bool)
    keep[moved] = False
    sampled = np.zeros(len(case.z), bool)
    sampled[sel] = True
    nown = 0
    for c, (i, k) in enumerate(PAIRS):
        col = (tD[i:i + 1], sv[i:i + 1], rD[k:] if k < 0 else rD[k:k + 1])
        s2, d2, f2 = (r[0, 0] for r in grid8_eval(ub.Params(pq), *col, z2, case.lay))
        assert np.array_equal(res[2][c, keep], f2[keep]), f"{case}: flags differ hot/exact"
        pairs = ((res[0][c], s2, bars[0][c], bars[1][c]), (res[1][c], d2, bars[2][c], bars[3][c]))
        for a, b, ref, noise in pairs:
            assert np.array_equal(np.isnan(a[keep]), np.isnan(b[keep])), f"{case}: NaN pattern hot/exact"
        miss = np.zeros(len(case.z), bool)
        for a, b, ref, noise in pairs:
            with np.errstate(invalid="ignore"):
                bar = np.where(sampled, RTOL * ref + noise, RTOL * np.abs(a))
                miss |= keep & ~(np.isnan(a) | (np.abs(a - b) <= bar) | (a == b))
        own = np.nonzero(miss & ~sampled)[0]
        if len(own):               # the oracle's own parity bar at these z
            pts = tuple(np.repeat(x, len(own)) for x in col) + (case.z[own], case.lay[own])
            so, do, sps, spd = oracle_with_noise(oracle.Params(pq), pts, points=True, nsamples=5)
            for (a, b, ref, noise), r, sp in zip(pairs, (so, do), (sps, spd)):
                ref[own], noise[own] = np.abs(r), NOISE_K * sp
            nown += len(own)
        for (a, b, ref, noise), what in zip(pairs, ("s", "ds")):
            with np.errstate(invalid="ignore"):
                bar = np.where(np.isnan(ref), RTOL * np.abs(a), RTOL * ref + noise)
            diff = np.abs(a - b)
            ok = ~keep | np.isnan(a) | (diff <= bar) | (a == b)
            assert ok.all(), (f"{case} {what} (t{i}, r{k}): hot vs exact, {int((~ok).sum())} points fail; worst "
                              f"rel {np.nanmax(np.where(ok, 0, diff / np.abs(a))):.3e}")
    return len(moved), nown


@pytest.mark.gpu
def test_designed_layouts_per_point_and_coverage(gpu):
    cases = designed_cases() + edge_cases()
    reached, reasons, wells, npts, nnudged, nown = set(), set(), [], 0, 0, 0
    for case in cases:
        res, sel, bars, well = run_case(case)      # every run of the case on lh_grid8_kernel (grid8_eval)
        npts += 2 * sel.size
        wells.append((well, str(case)))
        for c in case.cls:
            if c["reason"] is None:
                reached.add(hot_key(c))
            else:
                reasons.add(c["reason"])
        if case.nudge:
            nb, no = hot_vs_exact(case, res, sel, bars)
            nnudged, nown = nnudged + nb, nown + no
    wf = np.array([w for w, _ in wells])
    print(f"\n{len(cases)} cases, {npts} oracle points, {nnudged} blocks hot against exact "
          f"({nown} unsampled z held to their own oracle bar), "
          f"well-conditioned fraction {wf.mean():.3f}")
    print("least well-conditioned cases:", ", ".join(f"{n} {w:.2f}" for w, n in sorted(wells)[:6]))
    print("hot (kx, K0Z, Lb direction):", sorted(reached))
    print("slow-path reasons:", sorted(reasons))
    # the 1e-9 bar binds: most sampled points are well conditioned
    assert wf.mean() > 0.9, wf.mean()
    assert all(w >= 0.55 for w, _ in wells), [(n, w) for w, n in wells if w < 0.55]
    want = {(kx, k0z) for kx in (-1, 1, 2, 3, 4, 5, 6, 7) for k0z in (True, False)}
    got = {(kx, k0z) for kx, k0z, dirn in reached if kx == -1 or dirn != 0}
    assert want <= got, f"hot path not reached for {sorted(want - got)}"
    assert {dirn for kx, k0z, dirn in reached if kx >= 0} >= {1, -1}
    assert {(kx, k0z, -1) for kx, k0z, dirn in reached if kx == 7 and dirn == -1} == {(7, True, -1), (7, False, -1)}
    assert reasons == {"tail of 16 z or fewer", "not equally spaced", "several slots off the common layer",
                       "exception slot on two other layers"}


@pytest.mark.gpu
@pytest.mark.parametrize("nz", [40, 129, 150])
def test_carry_through_padded_grid8_items(gpu, nz):
    """Stale-infint carry (reference-compatible mode) through lh_grid8_kernel on items with padding
    slots: overflowing radii after healthy ones, over two times (driver.f90:205-214)."""
    d, pd = load_deck("hantush-contours-input.dat")
    rD = np.array([0.5, 0.2, 1e-3, 0.075, 5e-3, 0.02, 1.5, 2e-3])
    tD = np.array([d["tD"][0], 3.0 * d["tD"][0]])
    sv = oracle.split_index(tD, d["j0s"])
    zD = np.linspace(0.0, 1.0, nz)
    lay = oracle.zlay(zD, pd["lD"], pd["dD"])
    sc = float(d["j0z"][sv[0] - 1] / rD[0])
    sg, dg, fg = grid8_eval(ub.Params(pd), tD, sv, rD, zD, lay, ts_scale=sc)
    # the oracle's carry is per z: sample the ends of every slot of every block and the layer changes
    case = Case(f"carry-nz{nz}", "hantush-contours-input.dat", zD, lay)
    sel = oracle_sample(case)
    args = (tD, sv, rD, zD[sel], lay[sel])
    po = oracle.Params(pd)
    so, do, sps, spd = oracle_with_noise(po, args, ts_scale=sc, carry=True, nsamples=3)
    _, _, fo = oracle.eval_grid(po, *args, ts_scale=sc, carry=True)
    assert np.array_equal(fo, fg[:, :, sel])
    assert fo.any() and not fo.all()
    check_parity(sg[:, :, sel], dg[:, :, sel], so, do, sps, spd, what=f"carry nz={nz}")
    assert any(n < ZB for _, n in blocks(nz))      # some item has padding slots


@pytest.mark.gpu
def test_descending_block_small_radius(gpu):
    """A full descending block, boundary in slot 7 (Lb below Lc), at radii where Re(eta) comes near
    fast_eta_max: spx = cp(Lb) e^{eta D kx} with D < 0 is formed before the factor e^{eta z_first}.
    The largest Re(eta) = Re sqrt((p + a^2)/kappa) of the quadrature (a at the end of the last
    Gauss-Lobatto interval, every de Hoog p) must pass fast_eta_max = 700 / m (fast.cuh), so that
    the abscissae run on the hot path right up to the bound and the literal path beyond it."""
    _, pq, tD, sv = deck_of(DECKS[3])
    z, lay = boundary_list(pq, 3, 2, 7 * GL + 8, 128)
    z2, lay2 = boundary_list(pq, 2, 1, 7 * GL + 8, 128)
    for zz, ll in ((z, lay), (z2, lay2)):
        case = Case("moench:desc-small-rD", DECKS[3], zz, ll, rD=(0.035, 0.06))
        assert case.cls[0]["reason"] is None and case.cls[0]["kx"] == 7 and case.cls[0]["Lb"] < case.cls[0]["Lc"]
        m = max(1.0 + pq["dD"], float(np.float32(np.float32(np.abs(zz).max()) * np.float32(1.0000002))))
        assert pq["model"] == 3        # m = 1 + dD for models 3 and 5 (fast_eta_max)
        for i, r in zip((0, 1), case.rD):
            a = pq["j0z"][sv[i] + pq["gl_nacc"] - 1] / r
            p = oracle.pvalues(oracle.Params(pq), pq.get("tee_mult", 2.0) * tD[i])
            ratio = np.sqrt((p + a * a) / pq["kappa"]).real.max() / (700.0 / m)
            print(f"\n{case} rD = {r}: max Re(eta) / fast_eta_max = {ratio:.2f}")
            assert 1.0 < ratio < 3.0, ratio
        run_case(case)
