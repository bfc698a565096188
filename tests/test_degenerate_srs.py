"""Trapdoor checks of the MSM and KZG paths on degenerate and random SRSs, independent of every MSM.

For an SRS B_i = beta^i * G:   commit(p) = p(beta) * G   and   witness(p, z) = ((p(beta) - p(z)) / (beta - z)) * G.
The reference is one Horner evaluation (orc.fr_eval) and one scalar multiplication (orc.g1_mul), so it is cheap at any size.

A beta of small multiplicative order (0, 1, -1, w_4, w_256) makes the SRS a short period tiled to length n: every Pippenger
bucket then meets copies of a point or of its negative, and the batched-affine pair rounds (msm_affine.cuh) carry exceptional
pairs (P + P, P + (-P), identity operands) at every position of every thread's chain.  beta = +-2^c, with c the window of the
folded tables, makes table group k of base i equal to base i + k (up to sign), so the window folding itself collides.

Every case body takes (eng, pc, size, ...).  The CPU tests run the bodies on the kernels compiled for the host (tests/host_emul)
at reduced sizes: there a pair kernel has 48 threads, so the chains are long anyway.  The `gpu` tests run them on the device at
shapes where every pair-round thread carries several slots whatever the occupancy (asserted on the shape, `assert_long_chains`).
"""
import contextlib
import os

import numpy as np
import pytest

from oracle import orc, pyref
from tests import util

BETAS = ["0", "1", "-1", "w4", "w256", "2^c", "-2^c"]
FAMILIES = ["uniform", "equal", "pm1", "repeated"]
PAIR_T_CAP = 1 << 20       # msm.cuh caps a pair-round launch at 2^20 threads (a full resident wave is ~75 k on a B200)
PERIOD_MAX = 1 << 13       # longer periods are computed as plain powers


@contextlib.contextmanager
def env(**kv):
    """PCGPU_* knobs for the calls inside the block (the library reads them on every call)."""
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.fixture(scope="module")
def emu(pc, hostcheck_path):
    e = pc.Engine(0, lib_path=hostcheck_path)
    yield e
    e.close()


# ---- reference (no MSM anywhere) ---------------------------------------------------------------------------------------------
def beta_value(C, name, c):
    return {"0": 0, "1": 1, "-1": C.r - 1, "w4": C.domain_generator(2), "w256": C.domain_generator(8),
            "2^c": 1 << c, "-2^c": C.r - (1 << c)}[name]


def srs_of_order(cname, beta, n, eng=None):
    """B_i = beta^i * G for i < n -> ((n, 2*nq) uint64, (n,) uint8 identity flags).  One period of the powers is multiplied out
    on the host (orc.fixed_base_batch_mul) and tiled; beta = 0 gives [G, O, O, ...].  A period longer than PERIOD_MAX is
    computed in full, on the device when `eng` is given (spot-checked against the oracle)."""
    C = pyref.Curve(cname)
    G = orc.g1_generator(C.id)
    pows, x = [], 1
    while len(pows) < min(n, PERIOD_MAX):
        pows.append(x)
        x = x * beta % C.r
        if x in (0, 1):
            break
    if len(pows) < n and x not in (0, 1):                       # long period: all n powers
        canon = orc.fr_powers_canonical(C.id, C.fr_to_limbs([beta], True)[0], n)
        if eng is None:
            return orc.fixed_base_batch_mul(C.id, G, canon)
        xy = eng.fixed_base_mul(C.id, G, canon)
        idx = np.unique(np.concatenate([[0, 1, n - 1], util.rng(n).integers(0, n, size=8)]))
        assert (xy[idx] == orc.fixed_base_batch_mul(C.id, G, canon[idx])[0]).all()
        return xy, np.zeros(n, dtype=np.uint8)
    head, period = ([], pows) if x == 1 else (pows, [0])      # beta = 0: [1] then 0 forever
    if len(pows) >= n:
        head, period = pows[:n], []
    pts, inf = orc.fixed_base_batch_mul(C.id, G, C.fr_to_limbs(head + period, False))
    h = len(head)
    if not period:
        return pts, inf
    reps = -(-(n - h) // len(period))
    xy = np.concatenate([pts[:h], np.tile(pts[h:], (reps, 1))])[:n]
    return np.ascontiguousarray(xy), np.concatenate([inf[:h], np.tile(inf[h:], reps)])[:n].copy()


def to_mont(C, canon):
    return orc.field_unop("orc_fr_to_mont", C.id, canon) if len(canon) else canon


def p_at(C, coeffs_mont, x):
    """p(x) as an integer, for Montgomery coefficients (Horner in the C oracle)"""
    if len(coeffs_mont) == 0:
        return 0
    return C.fr_from_limbs(orc.fr_eval(C.id, coeffs_mont, C.fr_to_limbs([x], True)[0]), True)[0]


def g_mul(C, k):
    return orc.g1_mul(C.id, orc.g1_generator(C.id), C.fr_to_limbs([k % C.r], False)[0])


def ref_commit(C, coeffs_mont, beta):
    """commit(p) = p(beta) * G"""
    return g_mul(C, p_at(C, coeffs_mont, beta))


def ref_witness(C, coeffs_mont, beta, z):
    """witness(p, z) = ((p(beta) - p(z)) / (beta - z)) * G"""
    return g_mul(C, (p_at(C, coeffs_mont, beta) - p_at(C, coeffs_mont, z)) * pow(beta - z, -1, C.r))


def ref_msm_signed(C, points, j, e, s_mont):
    """Bases e_i * P_{j(i)} with e_i in {-1, 0, +1} (0: the identity base); scalars s (rows, cnt, 4) Montgomery.  Per row
    sum_j (sum_i e_i s_i) * P_j, the inner sums by the oracle's Fr row product -> list of (xy, inf)."""
    rows, cnt = s_mont.shape[0], s_mont.shape[1]
    st = np.ascontiguousarray(s_mont.transpose(1, 0, 2))                    # (cnt, rows, 4)
    lut = C.fr_to_limbs([0, 1, C.r - 1], True)
    coef = []
    for k in range(points.shape[0]):
        mask = lut[np.where(j == k, e, 0) % 3]                              # 0 -> 0, 1 -> 1, -1 -> r - 1
        coef.append(C.fr_from_limbs(orc.fr_row_mul(C.id, mask, st, cnt, rows), True))
    out = []
    for r in range(rows):
        terms = [orc.g1_mul(C.id, points[k], C.fr_to_limbs([coef[k][r]], False)[0]) for k in range(points.shape[0])]
        out.append(orc.g1_sum(C.id, np.stack([t[0] for t in terms]), inf=np.array([t[1] for t in terms], dtype=np.uint8)))
    return out


def scalars_of(cname, family, n, seed):
    """(n, 4) canonical scalars: uniform; all equal; {0, +-1}; or 80 % drawn from five values (heavy buckets)"""
    C = pyref.Curve(cname)
    g = util.rng(seed)
    if family == "uniform":
        return util.rand_fr(cname, n, seed, mont=False)
    if family == "equal":
        return np.tile(util.rand_fr(cname, 1, seed, mont=False), (n, 1))
    if family == "pm1":
        return C.fr_to_limbs([0, 1, C.r - 1], False)[g.integers(0, 3, size=n)]
    v = util.rand_fr_ints(cname, 1, seed)[0]
    sc = util.rand_fr(cname, n, seed + 1, mont=False)
    pick = g.integers(0, 5, size=n)
    heavy = g.random(n) < 0.8
    sc[heavy] = C.fr_to_limbs([1, C.r - 1, 2, v, C.r - v], False)[pick[heavy]]
    return sc


def pick_c(n):
    """msm.cuh msm_pick_c: the raw-base window"""
    return min(16, max(8, n.bit_length() - 1 - 4))


def assert_long_chains(C, n, c, tdiv):
    """Every thread of round 0 carries >= 4 slots whatever the occupancy: uniform scalars give about n*W entries, so at least
    n*(W-1)/2 pair slots (one window may be sparse), against at most PAIR_T_CAP / tdiv threads."""
    W = -(-C.r.bit_length() // c)
    slots = n * (W - 1) // 2
    assert slots >= 4 * PAIR_T_CAP // tdiv, (n, c, W, slots, tdiv)


def same(got, exp, what):
    xy, inf = got
    assert int(inf) == exp[1] and (exp[1] or (xy == exp[0]).all()), what


# ---- case bodies ---------------------------------------------------------------------------------------------------------------
def case_msm_paths(eng, pc, size, cname, beta_name, family, c, paths, tdiv=1):
    """one degenerate SRS of `size` bases, one scalar family, every listed MSM path against p(beta) * G"""
    C = pyref.Curve(cname)
    beta = beta_value(C, beta_name, c)
    bases, inf = srs_of_order(cname, beta, size, eng=eng if size > PERIOD_MAX else None)
    sc = scalars_of(cname, family, size, seed=100 * util.CURVE_NAMES.index(cname) + 10 * BETAS.index(beta_name) + FAMILIES.index(family))
    scm = to_mont(C, sc)
    exp = ref_commit(C, scm, beta)
    knobs = {"PCGPU_MSM_AFFINE_TDIV": tdiv} if tdiv > 1 else {}
    raw = eng.srs_register(C.id, bases, inf=inf)
    try:
        if "small" in paths:
            k = min(size, 4096)
            with env(PCGPU_MSM_SMALL=1):
                same(eng.msm(raw, sc[:k]), ref_commit(C, scm[:k], beta), "small")
                same(eng.msm(raw, scm[:k], flags=pc.SCALARS_MONT), ref_commit(C, scm[:k], beta), "small mont")
        for R in (0, 1, 3, 5):
            if f"rounds{R}" in paths:
                with env(PCGPU_MSM_SMALL=0, PCGPU_MSM_AFFINE_ROUNDS=R, **knobs):
                    same(eng.msm(raw, sc), exp, f"rounds {R}")
        if "c18" in paths:
            with env(PCGPU_MSM_SMALL=0, PCGPU_MSM_C=18):
                same(eng.msm(raw, sc), exp, "two-level reduction")
        if "partial" in paths:
            cuts = [0, size // 5, size // 2, size - 1, size]
            with env(PCGPU_MSM_SMALL=0):
                parts = [eng.msm_partial(raw, sc[a:b], base_offset=a) for a, b in zip(cuts[:-1], cuts[1:])]
            same(eng.g1_sum_xyzz(C.id, np.concatenate(parts)), exp, "partial")
        if "bases" in paths:
            with env(PCGPU_MSM_SMALL=0):
                same(eng.msm_bases(C.id, bases, scm, inf=inf, flags=pc.SCALARS_MONT), exp, "unregistered bases")
    finally:
        raw.release()
    if "folded" in paths:
        with env(PCGPU_SRS_C=c):                                  # pinned: beta = +-2^c is the folding window
            tab = eng.srs_register(C.id, bases, inf=inf, flags=pc.SRS_PRECOMPUTE)
        try:
            with env(PCGPU_MSM_SMALL=0):
                same(eng.msm(tab, sc), exp, "folded tables")
            with env(PCGPU_MSM_SMALL=0, PCGPU_MSM_AFFINE_ROUNDS=3, **knobs):
                same(eng.msm(tab, scm, flags=pc.SCALARS_MONT), exp, "folded tables, 3 rounds")
                off = 3
                exp_off = g_mul(C, p_at(C, scm[off:], beta) * pow(beta, off, C.r))      # &bases[off..]: beta^off * sum s_i beta^(i-off)
                same(eng.msm(tab, sc[off:], base_offset=off), exp_off, "folded tables, offset")
        finally:
            tab.release()


def case_comb_batch(eng, pc, size, cname, rows, seed):
    """msm_batch over SRS_COMB tables whose bases are duplicated, negated and identity copies of a few generators (Hyrax's
    row commitments over such a key), per row against ref_msm_signed"""
    C = pyref.Curve(cname)
    gens = util.random_points(cname, 3, seed=seed)
    g = util.rng(seed)
    j = g.integers(0, 3, size=size)
    e = g.choice([-1, 0, 1, 1], size=size)
    py = C.points_from_limbs(gens)
    bases, inf = C.points_to_limbs([None if ei == 0 else (py[ji] if ei > 0 else C.neg(py[ji])) for ji, ei in zip(j, e)])
    mat = util.rand_fr(cname, rows * size, seed + 1, mont=True).reshape(rows, size, 4)
    mat[1] = mat[0]                                               # two equal rows
    mat[2, :, :] = 0; mat[2, ::2] = util.fr_const(cname, 1)      # {0, 1} row
    exp = ref_msm_signed(C, gens, j, e, mat)
    srs = eng.srs_register(C.id, bases, inf=inf, flags=pc.SRS_COMB)
    try:
        got, ginf = eng.msm_batch(srs, mat, size, rows, flags=pc.SCALARS_MONT)
    finally:
        srs.release()
    for r in range(rows):
        same((got[r], ginf[r]), exp[r], ("comb row", r))


def kzg_polys(cname, size):
    """distinct polynomials of different lengths: full, trailing zeros, one coefficient, zero, and shorter ones"""
    polys = [util.rand_fr_fast(cname, size, seed=700), util.rand_fr_fast(cname, size, seed=701),
             util.rand_fr_fast(cname, 1, seed=702), np.zeros((5, 4), dtype=np.uint64),
             util.rand_fr_fast(cname, size // 2 + 7, seed=703), util.rand_fr_fast(cname, min(size, 4097), seed=704),
             util.rand_fr_fast(cname, min(size, 3000) - 1, seed=705)]
    polys[1][-(size // 7):] = 0
    return polys


def case_kzg_entry_points(eng, pc, size, cname, bases, beta, flags, combos):
    """kzg_commit / open / commit_open / commit_batch / commit_open_batch (host and device-resident coefficients, every
    (ways, tdiv) in `combos`) slot by slot against the trapdoor formulas"""
    C = pyref.Curve(cname)
    z = util.rand_fr(cname, 1, seed=710, mont=True)[0]
    zi = C.fr_from_limbs(z, True)[0]
    polys = kzg_polys(cname, size)
    exp_c = [ref_commit(C, p, beta) for p in polys]
    exp_w = [ref_witness(C, p, beta, zi) for p in polys]
    srs = eng.srs_register(C.id, bases, flags=flags)
    bufs = []
    try:
        for i in (0, 1, 4):
            same(eng.kzg_commit(srs, polys[i]), exp_c[i], ("commit", i))
            w = eng.kzg_open(srs, polys[i], z)
            same(w[:2], exp_w[i], ("open", i))
            (c, ci), (w, wi) = eng.kzg_commit_open(srs, polys[i], z)
            same((c, ci), exp_c[i], ("commit_open c", i))
            same((w, wi), exp_w[i], ("commit_open w", i))
        order = [0, 2, 1, 3, 4]
        got, ginf = eng.kzg_commit_batch(srs, [polys[i] for i in order])
        for k, i in enumerate(order):
            same((got[k], ginf[k]), exp_c[i], ("commit_batch", i))
        for p in polys:
            d = eng.buffer(p.shape[0])
            d.write(p)
            bufs.append(d)
        dev = [(d.ptr(), p.shape[0]) for d, p in zip(bufs, polys)]
        for ways, tdiv in combos:
            with env(PCGPU_COMMIT_OPEN_WAYS=ways, PCGPU_BATCH_TDIV=tdiv):
                for src, fl in ((polys, 0), (dev, pc.DEVICE_PTRS)):
                    c, ci, w, wi = eng.kzg_commit_open_batch(srs, src, z, flags=fl)
                    for i in range(len(polys)):
                        same((c[i], ci[i]), exp_c[i], ("batch commit", ways, tdiv, fl, i))
                        same((w[i], wi[i]), exp_w[i], ("batch witness", ways, tdiv, fl, i))
    finally:
        for d in bufs:
            d.release()
        srs.release()


# ---- CPU: the kernels compiled for the host --------------------------------------------------------------------------------
EMU_N, EMU_C = 1200, 12          # EMU_C: the folded-table window at n = 4200 (srs.cuh), pinned where tables are built


@pytest.mark.parametrize("cname", util.CURVE_NAMES)
@pytest.mark.parametrize("beta_name", BETAS)
def test_degenerate_srs_emulated(emu, pc, cname, beta_name):
    """each beta on each curve, the scalar family rotating so that every beta meets three of the four (beta = 1 with equal
    coefficients: every round-0 pair is a doubling), through the small path, 0 / 1 / 3 / 5 pair rounds, the two-level reduction,
    partial sums and unregistered bases"""
    fam = FAMILIES[(BETAS.index(beta_name) + util.CURVE_NAMES.index(cname)) % 4]
    case_msm_paths(emu, pc, EMU_N, cname, beta_name, fam, EMU_C,
                   ("small", "rounds0", "rounds1", "rounds3", "rounds5", "c18", "partial", "bases"))


@pytest.mark.parametrize("cname,beta_name,family", [("bn254", "2^c", "uniform"), ("pallas", "-2^c", "repeated"),
                                                    ("pallas", "1", "equal"), ("bn254", "w256", "pm1"),
                                                    ("bls12_381", "0", "uniform")])
def test_degenerate_srs_folded_emulated(emu, pc, cname, beta_name, family):
    """window-folded tables (n >= 4096) on a degenerate SRS, default and forced rounds"""
    case_msm_paths(emu, pc, 4200, cname, beta_name, family, EMU_C, ("folded",))


@pytest.mark.parametrize("cname", ["bn254", "bls12_381"])
def test_comb_batch_signed_generators_emulated(emu, pc, cname):
    case_comb_batch(emu, pc, 40, cname, rows=6, seed=720)


@pytest.mark.parametrize("beta_name", ["rand", "-1"])
def test_kzg_trapdoor_emulated(emu, pc, beta_name):
    cname, n = "bls12_381", 300
    C = pyref.Curve(cname)
    beta = C.r - 1 if beta_name == "-1" else util.rand_fr_ints(cname, 1, 730)[0]
    bases, _ = srs_of_order(cname, beta, n)
    case_kzg_entry_points(emu, pc, n, cname, bases, beta, 0, [(1, 1), (4, 2)])


# ---- B200 ------------------------------------------------------------------------------------------------------------------
DEV_N = 40000                    # raw bases: c = 11, W = 24 -> ~480 k round-0 slots against <= 2^16 threads at tdiv 16
DEV_TDIV = 16


@pytest.mark.gpu
@pytest.mark.parametrize("cname", util.CURVE_NAMES)
@pytest.mark.parametrize("beta_name", BETAS)
def test_degenerate_srs_device(gpu_engine, pc, cname, beta_name):
    """the emulated case at device size: pair rounds forced on a sixteenth of the resident wave, so every thread's chain has
    >= 4 slots; folded tables with the window pinned to c = 14 (beta = +-2^14)"""
    C = pyref.Curve(cname)
    assert_long_chains(C, DEV_N, pick_c(DEV_N), DEV_TDIV)
    fam = FAMILIES[(BETAS.index(beta_name) + util.CURVE_NAMES.index(cname)) % 4]
    case_msm_paths(gpu_engine, pc, DEV_N, cname, beta_name, fam, 14,
                   ("small", "rounds0", "rounds1", "rounds3", "rounds5", "c18", "partial", "bases", "folded"), tdiv=DEV_TDIV)


@pytest.mark.gpu
@pytest.mark.parametrize("cname", util.CURVE_NAMES)
@pytest.mark.parametrize("beta_name", ["1", "-1", "w256", "2^c"])
def test_long_chains_folded_device(gpu_engine, pc, cname, beta_name):
    """n = 2^20 + 1 on window-folded tables (c = 17, W = 15: ~7.9 M round-0 slots, >= 7 per thread for any wave) with the
    default number of rounds; beta = 1 also with all coefficients equal"""
    C = pyref.Curve(cname)
    n, c = (1 << 20) + 1, 17
    assert_long_chains(C, n, c, 1)
    beta = beta_value(C, beta_name, c)
    bases, inf = srs_of_order(cname, beta, n, eng=gpu_engine)
    with env(PCGPU_SRS_C=c):
        tab = gpu_engine.srs_register(C.id, bases, inf=inf, flags=pc.SRS_PRECOMPUTE)
    try:
        for fam in ("uniform", "equal") if beta_name == "1" else ("uniform",):
            sc = scalars_of(cname, fam, n, seed=740)
            same(gpu_engine.msm(tab, sc), ref_commit(C, to_mont(C, sc), beta), (fam, "folded 2^20"))
    finally:
        tab.release()


@pytest.mark.gpu
def test_comb_batch_signed_generators_device(gpu_engine, pc):
    case_comb_batch(gpu_engine, pc, 1025, "bn254", rows=64, seed=750)


@pytest.fixture(scope="module")
def cfg2_srs(gpu_engine):
    from tests.test_gpu_parity import gpu_srs, gpu_srs_beta
    cname, n = "bls12_381", (1 << 20) + 1
    C = pyref.Curve(cname)
    return C.fr_from_limbs(gpu_srs_beta(cname, 21), True)[0], gpu_srs(gpu_engine, cname, n, seed=21)


ALL_COMBOS = [(w, t) for w in (1, 2, 4) for t in (1, 2, 4)]


@pytest.mark.gpu
def test_kzg_trapdoor_random_beta_device(gpu_engine, pc, cfg2_srs):
    """the KZG entry points at the cfg2 size (2^20 + 1 powers, BLS12-381, folded tables) on a random-beta SRS"""
    beta, bases = cfg2_srs
    case_kzg_entry_points(gpu_engine, pc, bases.shape[0], "bls12_381", bases, beta, pc.SRS_PRECOMPUTE, ALL_COMBOS)


@pytest.mark.gpu
def test_kzg_trapdoor_beta_minus_one_device(gpu_engine, pc):
    """the same with beta = -1: the half-wave batch chains meet P + P and P + (-P) in every bucket"""
    cname, n = "bls12_381", (1 << 20) + 1
    C = pyref.Curve(cname)
    bases, _ = srs_of_order(cname, C.r - 1, n)
    case_kzg_entry_points(gpu_engine, pc, n, cname, bases, C.r - 1, pc.SRS_PRECOMPUTE, ALL_COMBOS)


@pytest.mark.gpu
def test_kzg_trapdoor_cfg5_shape_beta_minus_one_device(gpu_engine, pc):
    """cfg5's per-polynomial shape (2^22 + 1 powers, folded tables: 8 GB, released at the end) with beta = -1"""
    cname, n = "bls12_381", (1 << 22) + 1
    C = pyref.Curve(cname)
    bases, _ = srs_of_order(cname, C.r - 1, n)
    srs = gpu_engine.srs_register(C.id, bases, flags=pc.SRS_PRECOMPUTE)
    try:
        polys = [util.rand_fr_fast(cname, n, seed=760), util.rand_fr_fast(cname, n - 1000, seed=761)]
        exp = [ref_commit(C, p, C.r - 1) for p in polys]
        same(gpu_engine.kzg_commit(srs, polys[0]), exp[0], "cfg5 commit")
        got, ginf = gpu_engine.kzg_commit_batch(srs, polys)
        for i in range(2):
            same((got[i], ginf[i]), exp[i], ("cfg5 commit_batch", i))
    finally:
        srs.release()
