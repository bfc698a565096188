"""CPU unit tests of the DEVICE code compiled for the host (tests/host_emul): the production limb
schedule, digit recoding, bucket bookkeeping, scans and the C-ABI host logic, each against the C oracle
or the Python big-integer oracle.  These do not replace the GPU parity tests (tests/test_gpu_*.py); they
catch logic errors before GPU time is spent."""
import ctypes

import numpy as np
import pytest

from oracle import orc, pyref
from tests import golden_cases, util

FIELDS = [("bls12_381", "p", 0), ("bls12_381", "r", 1), ("bn254", "p", 2), ("bn254", "r", 3), ("pallas", "p", 4),
          ("pallas", "r", 5)]


@pytest.fixture(scope="module")
def eng(pc, hostcheck_path):
    e = pc.Engine(0, lib_path=hostcheck_path)
    yield e
    e.close()


def _tol(vs, n64):
    out = np.zeros((len(vs), n64), dtype=np.uint64)
    for i, v in enumerate(vs):
        for j in range(n64):
            out[i, j] = (v >> (64 * j)) & (2**64 - 1)
    return out


@pytest.mark.parametrize("cname,which,fid", FIELDS)
def test_field_schedule_vs_bigint(hostcheck_path, cname, which, fid):
    lib = ctypes.CDLL(hostcheck_path)
    C = pyref.Curve(cname)
    mod = getattr(C, which)
    n64 = (mod.bit_length() + 63) // 64
    R = (1 << (64 * n64)) % mod
    Rinv = pow(R, -1, mod)
    g = np.random.default_rng(fid)
    edge = [0, 1, 2, mod - 1, mod - 2, R, R * R % mod, mod >> 1, (mod >> 1) + 1, (1 << (mod.bit_length() - 1)),
            (1 << (mod.bit_length() - 1)) - 1, (1 << 32) - 1, (1 << 64) - 1, ((1 << (32 * 2 * n64 - 2)) - 1) % mod]
    rnd = [int.from_bytes(g.bytes(8 * n64), "little") % mod for _ in range(400)]
    va = edge + [e for e in edge for _ in edge] + rnd
    vb = edge + [e for _ in edge for e in edge] + rnd[::-1]
    A, B = _tol(va, n64), _tol(vb, n64)
    ops = [(0, lambda a, b: a * b * Rinv % mod), (1, lambda a, b: a * b * Rinv % mod), (2, lambda a, b: (a + b) % mod),
           (3, lambda a, b: (a - b) % mod), (4, lambda a, b: (-a) % mod), (6, lambda a, b: 0),
           (7, lambda a, b: (a * b + (a + b) * (b - a)) * Rinv % mod),   # 6, 7: sum of two products, one reduction
           (9, lambda a, b: a * a * Rinv % mod)]                          # dedicated squaring
    vp = ctypes.c_void_p
    for op, fn in ops:
        out = np.zeros_like(A)
        assert lib.hostcheck_field_op(fid, op, A.ctypes.data_as(vp), B.ctypes.data_as(vp), out.ctypes.data_as(vp),
                                      ctypes.c_size_t(len(va))) == 0
        exp = _tol([fn(a, b) for a, b in zip(va, vb)], n64)
        assert (out == exp).all(), (cname, which, op)
    k = 24
    out = np.zeros_like(A[:k])
    lib.hostcheck_field_op(fid, 5, A[:k].ctypes.data_as(vp), B[:k].ctypes.data_as(vp), out.ctypes.data_as(vp), ctypes.c_size_t(k))
    exp = _tol([(pow(a * Rinv % mod, -1, mod) * R % mod) if a else 0 for a in va[:k]], n64)
    assert (out == exp).all()
    # binary-GCD (almost Montgomery) inverse == Fermat inverse, on edge values and random ones
    k2 = 120
    sel = list(range(len(edge))) + list(range(len(va) - k2, len(va)))
    A2 = np.ascontiguousarray(A[sel]); out = np.zeros_like(A2)
    lib.hostcheck_field_op(fid, 8, A2.ctypes.data_as(vp), A2.ctypes.data_as(vp), out.ctypes.data_as(vp), ctypes.c_size_t(len(sel)))
    exp = _tol([(pow(va[i] * Rinv % mod, -1, mod) * R % mod) if va[i] else 0 for i in sel], n64)
    assert (out == exp).all()


@pytest.mark.parametrize("cname", util.CURVE_NAMES)
@pytest.mark.parametrize("n", [0, 1, 2, 33, 300])
def test_msm_vs_oracle(eng, pc, cname, n, msm_path):
    C = pyref.Curve(cname)
    bases = util.random_points(cname, max(n, 1) + 7, seed=n)
    srs = eng.srs_register(C.id, bases)
    sc = util.rand_fr(cname, n, seed=10 + n, mont=False)
    got = eng.msm(srs, sc, n=n)
    exp = orc.msm(C.id, bases, sc, n=n)
    assert got[1] == exp[1] and (got[0] == exp[0]).all()
    # Montgomery scalars (fused into_bigint) give the same point
    scm = orc.field_unop("orc_fr_to_mont", C.id, sc) if n else sc
    got2 = eng.msm(srs, scm, n=n, flags=pc.SCALARS_MONT)
    assert got2[1] == exp[1] and (got2[0] == exp[0]).all()
    # base_offset = &powers_of_g[k..]
    if n > 3:
        got3 = eng.msm(srs, sc[: n - 3], base_offset=5)
        exp3 = orc.msm(C.id, bases[5:], sc[: n - 3])
        assert (got3[0] == exp3[0]).all()


def test_msm_edge_scalars(eng, pc, msm_path):
    """zeros, ones, r-1, small values, repeated bases (P+P inside a bucket), P and -P cancelling."""
    cname = "bls12_381"
    C = pyref.Curve(cname)
    pts = util.random_points(cname, 8, seed=3)
    neg = C.points_to_limbs([C.neg(p) for p in C.points_from_limbs(pts[:2])])[0]
    bases = np.concatenate([pts, pts[:4], neg])  # 14 bases
    vals = [0, 1, C.r - 1, 2, 65535, 65536, (1 << 254), 12345, 0, 1, C.r - 1, 7, 0, 1]
    vals[12] = 0; vals[13] = 1  # pairs with base 1 (scalar 1): P + (-P) = O in bucket 1
    sc = C.fr_to_limbs(vals, False)
    srs = eng.srs_register(C.id, bases)
    got = eng.msm(srs, sc)
    exp = orc.msm(C.id, bases, sc, naive=True)
    assert got[1] == exp[1] and (got[0] == exp[0]).all()
    # all scalars equal -> one bucket per window holds every point
    sc2 = C.fr_to_limbs([0x1234567 for _ in range(14)], False)
    got = eng.msm(srs, sc2); exp = orc.msm(C.id, bases, sc2, naive=True)
    assert (got[0] == exp[0]).all()
    # result is the identity
    sc3 = C.fr_to_limbs([5, 0, 0, 0, 0, 0, 0, 0, C.r - 5, 0, 0, 0, 0, 0], False)
    got = eng.msm(srs, sc3)
    assert got[1] == 1 and not got[0].any()
    # out-of-range canonical scalar is rejected, not silently reduced
    bad = sc.copy(); bad[3, 3] = np.uint64(1 << 63)
    with pytest.raises(pc.PcgpuError) as ei:
        eng.msm(srs, bad)
    assert ei.value.code == -5
    # too many scalars for the bases
    with pytest.raises(pc.PcgpuError) as ei:
        eng.msm(srs, np.concatenate([sc, sc]))
    assert ei.value.code == -4


@pytest.mark.parametrize("rounds", [1, 3, 5])
def test_msm_batched_affine_rounds(eng, pc, rounds, monkeypatch):
    """msm_affine.cuh: forced batched-affine pairwise rounds (Montgomery batch inversion with the binary-GCD inverse)
    must give the same point, including the exceptional pairs: P + P, P + (-P), identity operands, odd bucket sizes."""
    monkeypatch.setenv("PCGPU_MSM_SMALL", "0")          # these cases target the bucket pipeline
    monkeypatch.setenv("PCGPU_MSM_AFFINE_ROUNDS", str(rounds))
    for cname, n in (("bls12_381", 150), ("bn254", 61), ("pallas", 90)):
        C = pyref.Curve(cname)
        pts = util.random_points(cname, n, seed=90 + rounds)
        neg = C.points_to_limbs([C.neg(p) for p in C.points_from_limbs(pts[:3])])[0]
        bases = np.concatenate([pts, pts[:5], neg])                 # repeated and negated bases
        inf = np.zeros(bases.shape[0], dtype=np.uint8); inf[7] = 1; inf[8] = 1
        sc = util.rand_fr(cname, bases.shape[0], seed=91 + rounds, mont=False)
        sc[n:n + 5] = sc[:5]                                        # same scalar on the repeated base -> P + P in a bucket
        sc[n + 5:] = sc[:3]                                         # same scalar on the negated base -> P + (-P)
        sc[20:40] = sc[20]                                          # a crowded bucket in every window
        srs = eng.srs_register(C.id, bases, inf=inf)
        got = eng.msm(srs, sc)
        exp = orc.msm(C.id, bases, sc, inf=inf)
        assert got[1] == exp[1] and (got[0] == exp[0]).all(), (cname, rounds)
    if rounds != 3:
        return
    # window-folded tables + rounds
    C = pyref.Curve("bn254")
    bases = util.random_points("bn254", 4200, seed=95)
    sc = util.rand_fr("bn254", 4200, seed=96, mont=False)
    srs = eng.srs_register(C.id, bases, flags=pc.SRS_PRECOMPUTE)
    got = eng.msm(srs, sc); exp = orc.msm(C.id, bases, sc)
    assert (got[0] == exp[0]).all()


@pytest.mark.parametrize("c", [18, 19])
def test_msm_two_level_reduction(eng, pc, c, monkeypatch):
    """large windows (c > 17): the weighted bucket sum goes through row / column sums (msm.cuh, h_split) -- forced here through
    the tuning knobs on the raw-base path and on window-folded tables."""
    monkeypatch.setenv("PCGPU_MSM_SMALL", "0")          # these cases target the bucket pipeline
    monkeypatch.setenv("PCGPU_MSM_C", str(c))
    monkeypatch.setenv("PCGPU_SRS_C", str(c))
    cname = "bn254"
    C = pyref.Curve(cname)
    n = 4200
    bases = util.random_points(cname, n, seed=97)
    sc = util.rand_fr(cname, n, seed=98, mont=False)
    sc[5] = C.fr_to_limbs([C.r - 1], False)[0]; sc[6] = 0; sc[7] = C.fr_to_limbs([1 << (c - 1)], False)[0]   # top bucket of window 0
    exp = orc.msm(C.id, bases, sc)
    srs = eng.srs_register(C.id, bases[:60])
    got = eng.msm(srs, sc[:60])
    assert (got[0] == orc.msm(C.id, bases[:60], sc[:60])[0]).all()
    if c == 18:
        srs = eng.srs_register(C.id, bases, flags=pc.SRS_PRECOMPUTE)
        got = eng.msm(srs, sc)
        assert (got[0] == exp[0]).all()


@pytest.mark.parametrize("rounds", ["0", "2"])
def test_msm_heavy_buckets(eng, pc, rounds, monkeypatch):
    """repeated scalars (many coefficients equal to 1, -1 or one constant -- common in real witness polynomials) put
    hundreds of points into single buckets: block-cooperative heavy-bucket reduction (MsmHeavyBucketBody)."""
    monkeypatch.setenv("PCGPU_MSM_SMALL", "0")          # these cases target the bucket pipeline
    monkeypatch.setenv("PCGPU_MSM_AFFINE_ROUNDS", rounds)
    cname = "bn254"
    C = pyref.Curve(cname)
    n = 1500
    bases = util.random_points(cname, n, seed=110)
    vals = [1] * 500 + [C.r - 1] * 400 + [0x1234567890abcdef1234567890abcdef] * 450 + util.rand_fr_ints(cname, 150, 111)
    sc = C.fr_to_limbs(vals, False)
    srs = eng.srs_register(C.id, bases)
    got = eng.msm(srs, sc)
    exp = orc.msm(C.id, bases, sc)
    assert got[1] == exp[1] and (got[0] == exp[0]).all()


def test_msm_infinity_bases(eng, msm_path):
    cname = "bn254"
    C = pyref.Curve(cname)
    pts = util.random_points(cname, 6, seed=4)
    inf = np.array([0, 1, 0, 0, 1, 0], dtype=np.uint8)
    sc = util.rand_fr(cname, 6, seed=5, mont=False)
    srs = eng.srs_register(C.id, pts, inf=inf)
    got = eng.msm(srs, sc)
    exp = orc.msm(C.id, pts, sc, inf=inf, naive=True)
    assert (got[0] == exp[0]).all()


def test_msm_precomputed_tables(eng, pc):
    """window folding: SRS_PRECOMPUTE tables must give the same point (n >= SRS_PRECOMPUTE_MIN_N path)."""
    cname = "bn254"
    C = pyref.Curve(cname)
    n = 4096 + 5
    bases = util.random_points(cname, n, seed=6)
    sc = util.rand_fr(cname, n, seed=7, mont=False)
    srs = eng.srs_register(C.id, bases, flags=pc.SRS_PRECOMPUTE)
    got = eng.msm(srs, sc)
    exp = orc.msm(C.id, bases, sc)
    assert (got[0] == exp[0]).all()
    got = eng.msm(srs, sc[:4090], base_offset=3)
    exp = orc.msm(C.id, bases[3:], sc[:4090])
    assert (got[0] == exp[0]).all()


@pytest.mark.parametrize("cname", ["bn254", "bls12_381"])
def test_msm_batch_shared_bases(eng, pc, cname):
    """HyraxPC::commit row loop (hyrax/mod.rs:233-242): dim Pedersen commitments over one com_key (+ h * r_i),
    comb tables and the no-table path, against one oracle MSM per row."""
    C = pyref.Curve(cname)
    dim = 9
    bases = util.random_points(cname, dim + 1, seed=50)       # com_key || h
    rows = util.rand_fr(cname, dim * (dim + 1), seed=51, mont=True).reshape(dim, dim + 1, 4)
    rows[2] = 0                                                # an all-zero row commits to the identity
    rows[3, :, :] = 0; rows[3, 0] = util.fr_const(cname, 1)    # = G_0
    canon = orc.field_unop("orc_fr_from_mont", C.id, rows.reshape(-1, 4)).reshape(dim, dim + 1, 4)
    exp = [orc.msm(C.id, bases, canon[r]) for r in range(dim)]
    for flags in (pc.SRS_COMB, 0):
        srs = eng.srs_register(C.id, bases, flags=flags)
        got, inf = eng.msm_batch(srs, rows, dim + 1, dim, flags=pc.SCALARS_MONT)
        for r in range(dim):
            assert inf[r] == exp[r][1] and (got[r] == exp[r][0]).all(), (flags, r)
        got2, _ = eng.msm_batch(srs, canon, dim + 1, dim)
        assert (got2 == got).all()
    assert inf[2] == 1


def test_kzg_commit_batch(eng, pc):
    """pcgpu_kzg_commit_batch (cfg5's shape: many polynomials over one SRS, 4 in flight) == one commit per polynomial."""
    cname = "bls12_381"
    C = pyref.Curve(cname)
    powers = util.synthetic_srs(cname, 65, seed=9)
    pg = eng.srs_register(C.id, powers)
    polys = [util.rand_fr(cname, 65 - (i % 3), seed=300 + i, mont=True) for i in range(7)]
    polys[2][:] = 0                                                        # a zero polynomial commits to the identity
    got, inf = eng.kzg_commit_batch(pg, polys)
    for i, p in enumerate(polys):
        rc, exy, einf = orc.kzg_commit(C.id, powers, p)
        assert rc == 0 and (got[i] == exy).all() and inf[i] == einf
    with pytest.raises(pc.PcgpuError) as ei:
        eng.kzg_commit_batch(pg, [util.rand_fr(cname, 80, seed=1, mont=True)])
    assert ei.value.code == -6


def test_kzg_commit_open_fused(eng, pc):
    """pcgpu_kzg_commit_open / _batch: one call == KZG10::commit then KZG10::open (kzg10/mod.rs:157-210, :287-310), including
    trailing zero coefficients, a constant and a zero polynomial, n beyond the small-MSM threshold, and the degree error"""
    cname = "bls12_381"
    C = pyref.Curve(cname)
    n = 4400
    powers = util.synthetic_srs(cname, n, seed=12)
    pg = eng.srs_register(C.id, powers, flags=pc.SRS_PRECOMPUTE)
    z = util.rand_fr(cname, 1, seed=401, mont=True)[0]
    polys = [util.rand_fr(cname, n, seed=400, mont=True), util.rand_fr(cname, 77, seed=402, mont=True),
             util.rand_fr(cname, 1, seed=403, mont=True), np.zeros((5, 4), dtype=np.uint64)]
    polys[0][-9:] = 0                                                       # trailing zeros are not part of the polynomial
    exp = []
    for p in polys:
        rc, cxy, cinf = orc.kzg_commit(C.id, powers, p)
        rc2, wxy, winf, _ = orc.kzg_open(C.id, powers, p, z)
        assert rc == 0 and rc2 == 0
        exp.append((cxy, cinf, wxy, winf))
        (c, ci), (w, wi) = eng.kzg_commit_open(pg, p, z)
        assert (c == cxy).all() and ci == cinf and (w == wxy).all() and wi == winf
    c, ci, w, wi = eng.kzg_commit_open_batch(pg, polys, z)
    for i, e in enumerate(exp):
        assert (c[i] == e[0]).all() and ci[i] == e[1] and (w[i] == e[2]).all() and wi[i] == e[3]
    with pytest.raises(pc.PcgpuError) as ei:
        eng.kzg_commit_open(pg, util.rand_fr(cname, n + 1, seed=404, mont=True), z)
    assert ei.value.code == -6
    # device-resident coefficients (the engine's own buffers: host memory under emulation): the trailing zeros must be trimmed
    # on the device side as well
    for p, e in zip(polys, exp):
        d = eng.buffer(p.shape[0])
        d.write(p)
        (c, ci), (w, wi) = eng.kzg_commit_open(pg, d.ptr(), z, n=p.shape[0], flags=pc.DEVICE_PTRS)
        assert (c == e[0]).all() and ci == e[1] and (w == e[2]).all() and wi == e[3]
        got = eng.kzg_commit(pg, d.ptr(), n=p.shape[0], flags=pc.DEVICE_PTRS)
        assert (got[0] == e[0]).all() and got[1] == e[1]
    d = eng.buffer(n + 50)                                                   # zero-filled
    d.write(polys[0])
    got = eng.kzg_commit(pg, d.ptr(), n=n + 50, flags=pc.DEVICE_PTRS)   # zero-padded beyond the SRS length: no E_DEGREE
    assert (got[0] == exp[0][0]).all()
    got = eng.kzg_open(pg, d.ptr(), z, n=n + 50, flags=pc.DEVICE_PTRS)
    assert (got[0] == exp[0][2]).all()


def test_marlin_pc_host_mirror(eng, pc):
    """marlin_pc.commit / open (mirror of marlin_pc/mod.rs:172-336) with and without degree bounds vs the oracle composed
    the same way: two_polys_degree_bound_single_query_test's shape (marlin_pc/mod.rs:720ff)."""
    from poly_commit_b200 import marlin_pc
    cname = "bls12_381"
    C = pyref.Curve(cname)
    max_degree, bounds = 40, [20, 33]
    pp = util.synthetic_srs(cname, max_degree + 1, seed=8)                 # universal powers_of_g[0..=max_degree]
    supported = 36
    powers = pp[: supported + 1]
    shifted = pp[max_degree - bounds[-1]:]                                   # trim(): powers_of_g[lowest_shift_degree..]
    ck = marlin_pc.CommitterKey(eng, C.id, powers, shifted, bounds)
    polys = [(util.rand_fr(cname, 30, seed=80, mont=True), None), (util.rand_fr(cname, 18, seed=81, mont=True), 20),
             (util.rand_fr(cname, 34, seed=82, mont=True), 33)]
    coms = marlin_pc.commit(ck, polys)
    for (coeffs, bound), (comm, sh) in zip(polys, coms):
        rc, exy, _ = orc.kzg_commit(C.id, powers, coeffs)
        assert rc == 0 and (comm[0] == exy).all()
        if bound is None:
            assert sh is None
        else:
            rc, sxy, _ = orc.kzg_commit(C.id, shifted[bounds[-1] - bound:], coeffs)
            assert rc == 0 and (sh[0] == sxy).all()
    point = util.rand_fr(cname, 1, seed=83, mont=True)[0]
    chals = util.rand_fr(cname, 5, seed=84, mont=True)
    w = marlin_pc.open(ck, polys, point, list(chals))
    # oracle composition of marlin_pc/mod.rs:245-336
    p = np.zeros((34, 4), dtype=np.uint64); sw = np.zeros((bounds[-1] + 1, 4), dtype=np.uint64); ci = 0
    for coeffs, bound in polys:
        p[: len(coeffs)] = orc.fr_axpy(C.id, p[: len(coeffs)], chals[ci], coeffs); ci += 1
        if bound is not None:
            wit, _ = orc.fr_div_linear(C.id, coeffs, point)
            s = np.concatenate([np.zeros((bounds[-1] - bound, 4), dtype=np.uint64), wit])
            sw[: len(s)] = orc.fr_axpy(C.id, sw[: len(s)], chals[ci], s); ci += 1
    rc, w0, _, _ = orc.kzg_open(C.id, powers, p, point)
    rc2, w1, _ = orc.kzg_commit(C.id, shifted, sw)
    exp, _ = orc.g1_sum(C.id, np.stack([w0, w1]))
    assert rc == 0 and rc2 == 0 and (w[0] == exp).all()
    with pytest.raises(ValueError):
        marlin_pc.commit(ck, [(polys[2][0], 20)])                            # bound below the degree
    # verifier side: Marlin::accumulate_commitments_and_values (marlin/mod.rs:109-148) on these commitments
    vals_int = [pyref.poly_eval(C.fr_from_limbs(c, True), C.fr_from_limbs(point, True)[0], C.r) for c, _ in polys]
    vals = C.fr_to_limbs(vals_int, True)
    shift_powers = {b: pp[max_degree - b] for b in bounds}                  # beta^(max_degree - bound) G
    triples = [(comm[0], None if sh is None else sh[0], bound) for (_, bound), (comm, sh) in zip(polys, coms)]
    (acc, ainf), cval = marlin_pc.accumulate_commitments_and_values(eng, C.id, triples, vals, list(chals), shift_powers)
    ch_int = C.fr_from_limbs(chals, True)
    exp_pt, exp_val, ci = None, 0, 0
    for (coeffs, bound), (comm, sh), v in zip(polys, coms, vals_int):
        cp = C.points_from_limbs(comm[0].reshape(1, -1))[0]
        exp_pt = C.add(exp_pt, C.mul(ch_int[ci], cp)); exp_val = (exp_val + ch_int[ci] * v) % C.r; ci += 1
        if bound is not None:
            sp = C.points_from_limbs(sh[0].reshape(1, -1))[0]
            shp = C.points_from_limbs(shift_powers[bound].reshape(1, -1))[0]
            exp_pt = C.add(exp_pt, C.mul(ch_int[ci], C.add(sp, C.neg(C.mul(v, shp))))); ci += 1
    ex, _ = C.points_to_limbs([exp_pt])
    assert not ainf and (acc == ex[0]).all() and C.fr_from_limbs(cval, True)[0] == exp_val


def test_marlin_pc_hiding_and_bounds(eng, pc):
    """MarlinKZG10::commit / open with hiding bounds AND degree bounds (marlin_pc/mod.rs:192-241, :245-336: r, shifted_r,
    shifted_r_witness, random_v) against the oracle composed step by step like the reference; accumulators device-resident."""
    from poly_commit_b200 import marlin_pc
    cname = "bls12_381"
    C = pyref.Curve(cname)
    max_degree, bounds = 40, [20, 33]
    pp = util.synthetic_srs(cname, max_degree + 1, seed=8)
    gamma = util.random_points(cname, 8, seed=85)                               # powers_of_gamma_g[0..=hiding_bound+1]
    supported = 36
    powers, shifted = pp[: supported + 1], pp[max_degree - bounds[-1]:]
    ck = marlin_pc.CommitterKey(eng, C.id, powers, shifted, bounds, powers_of_gamma_g_xy=gamma)
    polys = [(util.rand_fr(cname, 30, seed=80, mont=True), None), (util.rand_fr(cname, 18, seed=81, mont=True), 20),
             (util.rand_fr(cname, 34, seed=82, mont=True), 33), (util.rand_fr(cname, 9, seed=86, mont=True), None)]
    rands = [dict(rand=util.rand_fr(cname, 4, seed=87, mont=True)),
             dict(rand=util.rand_fr(cname, 5, seed=88, mont=True), shifted_rand=util.rand_fr(cname, 5, seed=89, mont=True)),
             dict(rand=util.rand_fr(cname, 3, seed=90, mont=True), shifted_rand=util.rand_fr(cname, 6, seed=91, mont=True)),
             None]                                                               # the last polynomial is committed without hiding
    coms = marlin_pc.commit(ck, polys, rands)
    for (coeffs, bound), rd, (comm, sh) in zip(polys, rands, coms):
        rc, exy, _ = orc.kzg_commit(C.id, powers, coeffs, gamma if rd else None, rd["rand"] if rd else None)
        assert rc == 0 and (comm[0] == exy).all()
        if bound is not None:
            rc, sxy, _ = orc.kzg_commit(C.id, shifted[bounds[-1] - bound:], coeffs, gamma, rd["shifted_rand"])
            assert rc == 0 and (sh[0] == sxy).all()
    point = util.rand_fr(cname, 1, seed=83, mont=True)[0]
    chals = util.rand_fr(cname, 6, seed=84, mont=True)
    w_xy, w_inf, random_v = marlin_pc.open(ck, polys, point, list(chals), rands)
    # the reference's composition on the oracle
    p = np.zeros((34, 4), dtype=np.uint64); r = np.zeros((6, 4), dtype=np.uint64)
    sw = np.zeros((bounds[-1] + 1, 4), dtype=np.uint64); sr = np.zeros((6, 4), dtype=np.uint64); ci = 0
    for (coeffs, bound), rd in zip(polys, rands):
        cj = chals[ci]; ci += 1
        p[: len(coeffs)] = orc.fr_axpy(C.id, p[: len(coeffs)], cj, coeffs)
        if rd:
            r[: len(rd["rand"])] = orc.fr_axpy(C.id, r[: len(rd["rand"])], cj, rd["rand"])
        if bound is not None:
            cj1 = chals[ci]; ci += 1
            wit, _ = orc.fr_div_linear(C.id, coeffs, point)
            s = np.concatenate([np.zeros((bounds[-1] - bound, 4), dtype=np.uint64), wit])
            sw[: len(s)] = orc.fr_axpy(C.id, sw[: len(s)], cj1, s)
            sr[: len(rd["shifted_rand"])] = orc.fr_axpy(C.id, sr[: len(rd["shifted_rand"])], cj1, rd["shifted_rand"])
    rc, w0, _, rv0 = orc.kzg_open(C.id, powers, p, point, gamma, r)
    srw, rv1 = orc.fr_div_linear(C.id, sr, point)
    rc2, w1, _ = orc.kzg_commit(C.id, shifted, sw, gamma, srw)                   # msm(shifted, shifted_w) + msm(gamma, shifted_r_witness)
    exp, _ = orc.g1_sum(C.id, np.stack([w0, w1]))
    assert rc == 0 and rc2 == 0 and not w_inf and (w_xy == exp).all()
    rv = (C.fr_from_limbs(rv0, True)[0] + C.fr_from_limbs(rv1, True)[0]) % C.r
    assert C.fr_from_limbs(random_v, True)[0] == rv
    # hiding without degree bounds: random_v is blind(point) of the combined blinding polynomial
    w2 = marlin_pc.open(ck, [polys[0], polys[3]], point, list(chals[:2]), [rands[0], None])
    p2 = np.zeros((30, 4), dtype=np.uint64)
    p2[:30] = orc.fr_axpy(C.id, p2[:30], chals[0], polys[0][0]); p2[:9] = orc.fr_axpy(C.id, p2[:9], chals[1], polys[3][0])
    r2 = orc.fr_axpy(C.id, np.zeros((4, 4), dtype=np.uint64), chals[0], rands[0]["rand"])
    rc, e2, _, erv = orc.kzg_open(C.id, powers, p2, point, gamma, r2)
    assert rc == 0 and (w2[0] == e2).all() and (w2[2] == erv).all()


def test_hyrax_host_mirror(eng, pc):
    """hyrax.commit / open_row_mul (mirror of hyrax/mod.rs:230-242, :347) vs the oracle, 4 variables -> dim 4."""
    from poly_commit_b200 import hyrax
    cname = "bn254"
    C = pyref.Curve(cname)
    dim = 4
    gens = util.random_points(cname, dim + 1, seed=60)
    ck = hyrax.CommitterKey(eng, C.id, gens[:dim], gens[dim])
    evals = util.rand_fr(cname, dim * dim, seed=61, mont=True)
    rnd = util.rand_fr(cname, dim, seed=62, mont=True)
    row_coms, inf, mat = hyrax.commit(ck, evals, rnd)
    assert (mat[1, 2] == evals[2 * dim + 1]).all()            # flat_to_matrix_column_major: row[r][c] = flat[c*n + r]
    for r in range(dim):
        sc = np.concatenate([mat[r], rnd[r:r + 1]])
        exp = orc.msm(C.id, gens, orc.field_unop("orc_fr_from_mont", C.id, sc))
        assert (row_coms[r] == exp[0]).all()
    l = util.rand_fr(cname, dim, seed=63, mont=True)
    lt = hyrax.open_row_mul(ck, mat, l)
    assert (lt == orc.fr_row_mul(C.id, l, mat.reshape(-1, 4), dim, dim)).all()
    pc0 = hyrax.pedersen_commit(ck, mat[0])
    assert (pc0[0] == orc.msm(C.id, gens[:dim], orc.field_unop("orc_fr_from_mont", C.id, mat[0]))[0]).all()
    # verifier side (hyrax/mod.rs:498-504): t_prime = <l, row_coms> must commit to lt with randomness <l, r>
    t_prime, tinf = hyrax.check_t_prime(eng, C.id, row_coms, l, inf)
    lr = eng.fr_inner_product(C.id, l, rnd)
    exp = orc.msm(C.id, gens, orc.field_unop("orc_fr_from_mont", C.id, np.concatenate([lt, lr.reshape(1, 4)])))
    assert (t_prime == exp[0]).all() and not tinf


@pytest.mark.parametrize("cname", util.CURVE_NAMES)
def test_msm_partial_and_sum(eng, cname):
    """index-range sharding (SURVEY 8e partitioning B): partial XYZZ sums add up to the whole MSM."""
    C = pyref.Curve(cname)
    n = 97
    bases = util.random_points(cname, n, seed=8)
    sc = util.rand_fr(cname, n, seed=9, mont=False)
    srs = eng.srs_register(C.id, bases)
    cuts = [0, 30, 30, 64, 97]  # includes an empty shard
    parts = [eng.msm_partial(srs, sc[a:b], n=b - a, base_offset=a) for a, b in zip(cuts[:-1], cuts[1:])]
    got = eng.g1_sum_xyzz(C.id, np.concatenate(parts))
    exp = orc.msm(C.id, bases, sc)
    assert (got[0] == exp[0]).all()


@pytest.mark.parametrize("cname", util.CURVE_NAMES)
def test_fixed_base_mul(eng, cname):
    C = pyref.Curve(cname)
    ks = util.rand_fr(cname, 20, seed=11, mont=False)
    ks[0] = 0
    ks[1] = C.fr_to_limbs([1], False)[0]
    got = eng.fixed_base_mul(C.id, orc.g1_generator(C.id), ks)
    exp, einf = orc.fixed_base_batch_mul(C.id, orc.g1_generator(C.id), ks)
    assert einf[0] == 1 and not got[0].any()
    assert (got[1:] == exp[1:]).all()


@pytest.mark.parametrize("cname", util.CURVE_NAMES)
@pytest.mark.parametrize("n,mode", [(1, "tile"), (2, "tile"), (31, "tree"), (32, "tile"), (33, "scan"), (2048, "tile"), (2049, "tile"),
                                    (2049, "tree"), (5000, "tree"), (6145, "tile"), (70001, "scan"), (70001, "tile"), (70001, "tree")])
def test_fr_div_linear(eng, cname, n, mode, monkeypatch):
    # tile: the one-pass kernel (tiles chained by a decoupled look-back; the default up to 2^21 coefficients), tree: the level
    # tree (the default beyond), scan: the one-block carry scan (kept as an experiment knob)
    monkeypatch.setenv("PCGPU_DIV_MODE", "tile" if mode == "tile" else "tree")
    if mode == "scan":
        monkeypatch.setenv("PCGPU_DIV_BLOCK_SCAN", "1")
    C = pyref.Curve(cname)
    p = util.rand_fr(cname, n, seed=20 + n, mont=True)
    z = util.rand_fr(cname, 1, seed=21, mont=True)[0]
    q, rem = eng.fr_div_linear(C.id, p, z)
    eq, erem = orc.fr_div_linear(C.id, p, z)
    assert (q == eq).all() and (rem == erem).all()
    assert (rem == orc.fr_eval(C.id, p, z)).all()


@pytest.mark.parametrize("cname", util.CURVE_NAMES)
def test_fr_vector_ops(eng, cname):
    C = pyref.Curve(cname)
    n = 777
    x = util.rand_fr(cname, n, seed=30, mont=True)
    y = util.rand_fr(cname, n, seed=31, mont=True)
    c = util.rand_fr(cname, 1, seed=32, mont=True)[0]
    assert (eng.fr_axpy(C.id, y, c, x) == orc.fr_axpy(C.id, y, c, x)).all()
    assert (eng.fr_from_mont(C.id, x) == orc.field_unop("orc_fr_from_mont", C.id, x)).all()
    assert (eng.fr_inner_product(C.id, x, y) == orc.fr_inner_product(C.id, x, y)).all()
    rows, cols = 13, 17
    m = util.rand_fr(cname, rows * cols, seed=33, mont=True)
    assert (eng.fr_row_mul(C.id, x[:rows], m, rows, cols) == orc.fr_row_mul(C.id, x[:rows], m, rows, cols)).all()


def test_row_mul_reference_kat(eng):
    """utils.rs:274-286 test_row_mul: [12, 41, 55] * [[10,100,4],[23,1,0],[55,58,9]] = [4088, 4431, 543]."""
    golden_cases.check_row_mul_kat(eng)


@pytest.mark.parametrize("cname", util.CURVE_NAMES)
def test_golden_vectors(eng, cname, msm_path):
    golden_cases.check_engine(eng, cname)
    golden_cases.check_wire_engine(eng, cname)


def oracle_ipa_rounds(cname, comm_key, coeffs, point, h_prime, round_challenge):
    """InnerProductArgPC::open's halving loop (ipa_pc/mod.rs:665-711) restated over the C oracle's primitives."""
    from poly_commit_b200 import ipa_pc
    C = pyref.Curve(cname)
    n = comm_key.shape[0]
    co = np.zeros((n, 4), dtype=np.uint64); co[: coeffs.shape[0]] = coeffs
    z_int = C.fr_from_limbs(point, True)[0]
    z = C.fr_to_limbs([pow(z_int, i, C.r) for i in range(n)], True)
    key = comm_key.copy()
    l_vec, r_vec = [], []
    while n > 1:
        m = n // 2
        def cm(keypart, sc, ip):
            msm, inf = orc.msm(C.id, keypart, orc.field_unop("orc_fr_from_mont", C.id, sc))
            hp, hinf = orc.g1_mul(C.id, h_prime, orc.field_unop("orc_fr_from_mont", C.id, ip.reshape(1, 4)))
            return orc.g1_sum(C.id, np.stack([msm, hp]), inf=np.array([inf, hinf], dtype=np.uint8))[0]
        l = cm(key[:m], co[m:n], orc.fr_inner_product(C.id, co[m:n], z[:m]))
        r = cm(key[m:n], co[:m], orc.fr_inner_product(C.id, co[:m], z[m:n]))
        l_vec.append(l); r_vec.append(r)
        # the reference's transcript, built independently of the device encoder: canonical LE scalar, then ark-serialize's
        # uncompressed encodings of l and r (oracle/pyref.py)
        data = int(round_challenge).to_bytes(32, "little") + pyref.g1_serialize(C, C.points_from_limbs(np.stack([l, r])), False)
        digest_i = 0
        while True:                                                   # compute_random_oracle_challenge, ipa_pc/mod.rs:74-87
            import hashlib
            v = int.from_bytes(hashlib.blake2s(data + digest_i.to_bytes(8, "little")).digest(), "little") % (1 << C.r.bit_length())
            if v < C.r:
                break
            digest_i += 1
        round_challenge = v
        inv = pow(round_challenge, -1, C.r)
        co[:m] = orc.fr_axpy(C.id, co[:m], C.fr_to_limbs([inv], True)[0], co[m:n])
        z[:m] = orc.fr_axpy(C.id, z[:m], C.fr_to_limbs([round_challenge], True)[0], z[m:n])
        key[:m] = orc.g1_fold(C.id, key[:n], C.fr_to_limbs([round_challenge], False))
        n = m
    return dict(l_vec=l_vec, r_vec=r_vec, final_comm_key=key[0], c=co[0])


@pytest.mark.parametrize("cname,n", [("pallas", 64), ("bls12_381", 16), ("bn254", 32)])
def test_ipa_open_rounds(eng, pc, cname, n, msm_path):
    """cfg3's dataflow (Pallas; the reference instantiates IPA on Jubjub only): every l, r, the final key and c."""
    from poly_commit_b200 import ipa_pc
    C = pyref.Curve(cname)
    key = util.random_points(cname, n, seed=70)
    h_prime = util.random_points(cname, 1, seed=71)[0]
    coeffs = util.rand_fr(cname, n - 3, seed=72, mont=True)     # fewer than d+1 coefficients: zero padded (:636-641)
    point = util.rand_fr(cname, 1, seed=73, mont=True)[0]
    got = ipa_pc.open_rounds(eng, C.id, key, coeffs, point, h_prime, 0x1234567)
    exp = oracle_ipa_rounds(cname, key, coeffs, point, h_prime, 0x1234567)
    assert len(got["l_vec"]) == n.bit_length() - 1
    for a, b in zip(got["l_vec"] + got["r_vec"], exp["l_vec"] + exp["r_vec"]):
        assert (a == b).all()
    assert (got["final_comm_key"] == exp["final_comm_key"]).all() and (got["c"] == exp["c"]).all()
    # verifier side (ipa_pc/mod.rs:760-766): cm_commit(comm_key, check_poly.compute_coeffs()) == proof.final_comm_key
    fk = ipa_pc.check_final_key(eng, C.id, key, got["challenges"])
    assert fk[1] == 0 and (fk[0] == got["final_comm_key"]).all()


@pytest.mark.parametrize("cname", util.CURVE_NAMES)
@pytest.mark.parametrize("logn,n_in", [(1, 2), (3, 5), (6, 64), (10, 700), (11, 2048), (12, 3000), (13, 8192)])
def test_ntt_vs_oracle(eng, cname, logn, n_in):
    """fft semantics of linear_codes/utils.rs:119-126 (zero-padded, natural order) and ifft(fft(x)) == x."""
    C = pyref.Curve(cname)
    x = util.rand_fr(cname, n_in, seed=300 + logn, mont=True)
    got = eng.ntt(C.id, x, logn)
    assert (got == orc.fr_ntt(C.id, x, logn)).all()
    back = eng.ntt(C.id, got, logn, inverse=True)
    assert (back[:n_in] == x).all() and not back[n_in:].any()


@pytest.mark.parametrize("cname", ["bls12_381", "bn254"])
def test_kzg_commit_open(eng, pc, cname, msm_path):
    """KZG10::commit / open dataflow (kzg10/mod.rs:157-310), non-hiding and hiding, vs the C oracle."""
    C = pyref.Curve(cname)
    n = 200
    powers = util.synthetic_srs(cname, n + 1, seed=1)
    gammas = util.random_points(cname, 8, seed=40)
    coeffs = util.rand_fr(cname, n, seed=41, mont=True)
    coeffs[0] = 0; coeffs[1] = 0          # leading (low-index) zeros: skip_leading_zeros path
    coeffs[n - 1] = 0                     # trailing zero: degree = n-2
    z = util.rand_fr(cname, 1, seed=42, mont=True)[0]
    pg, gg = eng.srs_register(C.id, powers), eng.srs_register(C.id, gammas)
    comm = eng.kzg_commit(pg, coeffs)
    rc, exy, einf = orc.kzg_commit(C.id, powers, coeffs)
    assert rc == 0 and (comm[0] == exy).all() and comm[1] == einf
    w = eng.kzg_open(pg, coeffs, z)
    rc, wxy, winf, _ = orc.kzg_open(C.id, powers, coeffs, z)
    assert rc == 0 and (w[0] == wxy).all()
    blind = util.rand_fr(cname, 3, seed=43, mont=True)
    comm = eng.kzg_commit(pg, coeffs, powers_of_gamma_g=gg, blind=blind)
    rc, exy, einf = orc.kzg_commit(C.id, powers, coeffs, gammas, blind)
    assert rc == 0 and (comm[0] == exy).all()
    w = eng.kzg_open(pg, coeffs, z, powers_of_gamma_g=gg, blind=blind)
    rc, wxy, winf, rv = orc.kzg_open(C.id, powers, coeffs, z, gammas, blind)
    assert rc == 0 and (w[0] == wxy).all() and (w[2] == rv).all()
    # degree too large -> TooManyCoefficients
    small = eng.srs_register(C.id, powers[:50])
    with pytest.raises(pc.PcgpuError) as ei:
        eng.kzg_commit(small, coeffs)
    assert ei.value.code == -6
    # constant and zero polynomials
    one = coeffs[:1].copy(); one[0] = util.fr_const(cname, 5)
    c1 = eng.kzg_commit(pg, one); rc, e1, _ = orc.kzg_commit(C.id, powers, one)
    assert (c1[0] == e1).all()
    w1 = eng.kzg_open(pg, one, z)
    assert w1[1] == 1  # witness of a constant is the zero polynomial -> identity
    zero = np.zeros((4, 4), dtype=np.uint64)
    c0 = eng.kzg_commit(pg, zero)
    assert c0[1] == 1


# ---- G1 wire formats (SURVEY 8f rank 1) -----------------------------------------------------------------------------
def _wire_points(cname, n, seed):
    C = pyref.Curve(cname)
    xy = util.random_points(cname, n, seed)
    pts = C.points_from_limbs(xy)
    # edge elements: identity, generator, -generator
    pts[0] = None
    pts[1] = C.g
    pts[2] = C.neg(C.g)
    xy2, inf = C.points_to_limbs(pts)
    return C, pts, xy2, inf


@pytest.mark.parametrize("cname", ["bls12_381", "bn254", "pallas"])
@pytest.mark.parametrize("compressed", [True, False])
def test_wire_roundtrip_vs_oracle(eng, cname, compressed):
    """serialize == the Python restatement byte for byte; deserialize(serialize(P)) == P with validation on
    (decompression square root, sign selection, on-curve and subgroup checks all exercised)."""
    C, pts, xy, inf = _wire_points(cname, 40, seed=61)
    assert eng.g1_wire_size(C.id, compressed) == pyref.wire_size(C, compressed)
    got = eng.g1_serialize(C.id, xy, inf, compressed)
    exp = pyref.g1_serialize(C, pts, compressed)
    assert got.tobytes() == exp
    back_xy, back_inf = eng.g1_deserialize(C.id, exp, len(pts), compressed, validate=True)
    assert (back_inf == inf).all() and (back_xy == xy).all()
    # the oracle's reader agrees with the device's on the same bytes
    assert pyref.g1_deserialize(C, got.tobytes(), len(pts), compressed) == pts
    # device convention: (0, 0) without an infinity byte is the identity as well
    assert eng.g1_serialize(C.id, xy, None, compressed).tobytes() == exp


def test_wire_bls12_381_generator_known_answer(eng):
    """the one published byte vector for this path: the ZCash compressed encoding of the BLS12-381 G1 generator"""
    C = pyref.Curve("bls12_381")
    kat = bytes.fromhex("97f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac58"
                        "6c55e83ff97a1aeffb3af00adb22c6bb")
    xy, inf = C.points_to_limbs([C.g])
    assert eng.g1_serialize(C.id, xy, inf, True).tobytes() == kat
    back, binf = eng.g1_deserialize(C.id, kat, 1, True)
    assert (back == xy).all() and not binf.any()
    assert eng.g1_serialize(C.id, xy, np.array([1], dtype=np.uint8), True).tobytes() == bytes([0xC0]) + bytes(47)


@pytest.mark.parametrize("cname", ["bls12_381", "bn254", "pallas"])
def test_wire_rejects_like_the_oracle(eng, pc, cname):
    """every failure class of CanonicalDeserialize: unexpected flags, non-canonical coordinate, x with no point, off-curve
    uncompressed point, (BLS12-381) on-curve point outside the prime-order subgroup -- the device reports the same first
    offending index and reason as the Python restatement, and Validate::No accepts what only validation rejects."""
    C, pts, xy, inf = _wire_points(cname, 12, seed=62)
    p = C.p
    zc = cname == "bls12_381"

    def both(data, n, compressed, validate=True):
        try:
            exp = pyref.g1_deserialize(C, data, n, compressed, validate)
            exp_err = None
        except pyref.WireError as e:
            exp, exp_err = None, (e.index, e.reason)
        try:
            got = eng.g1_deserialize(C.id, data, n, compressed, validate)
            got_err = None
        except pc.binding.WireError as e:
            got, got_err = None, (e.index, e.reason)
            assert e.code == pc.binding.E_INVALID
        assert got_err == exp_err, (cname, compressed, got_err, exp_err)
        if exp is not None:
            gx, gi = got
            ex, ei = C.points_to_limbs(exp)
            assert (gx == ex).all() and (gi == ei).all()
        return exp_err

    for compressed in (True, False):
        good = bytearray(pyref.g1_serialize(C, pts, compressed))
        sz = pyref.wire_size(C, compressed)
        assert both(bytes(good), len(pts), compressed) is None
        # (1) flags
        bad = bytearray(good)
        if zc:
            bad[5 * sz] ^= 0x80                              # compression bit contradicts the mode
        else:
            bad[6 * sz - 1] |= 0xC0                          # YIsNegative and PointAtInfinity together
        assert both(bytes(bad), len(pts), compressed) == (5, pyref.WIRE_BAD_FLAGS)
        # (2) x = p (not canonical)
        bad = bytearray(good)
        if zc:
            enc = bytearray(p.to_bytes(48, "big")); enc[0] |= 0x80 if compressed else 0
            bad[3 * sz:3 * sz + 48] = enc
        else:
            nb = (p.bit_length() + (2 if compressed else 0) + 7) // 8
            bad[3 * sz:3 * sz + nb] = p.to_bytes(nb, "little")
        assert both(bytes(bad), len(pts), compressed) == (3, pyref.WIRE_NOT_CANONICAL)
        # (3) no point with that x / y does not match x
        x = 1
        while pyref.fq_sqrt(C, x ** 3 + C.b) is not None:
            x += 1
        bad = bytearray(good)
        if compressed:
            one = pyref.g1_serialize(C, [(x, 0)], True)      # y only feeds the sign flag
        else:
            one = pyref.g1_serialize(C, [(pts[4][0], (pts[4][1] + 1) % p)], False)
        bad[4 * sz:5 * sz] = one
        assert both(bytes(bad), len(pts), compressed) == (4, pyref.WIRE_NOT_ON_CURVE)
        if not compressed:
            assert both(bytes(bad), len(pts), compressed, validate=False) is None
        # (4) on the curve, outside the subgroup (only BLS12-381 has a cofactor)
        if zc:
            Q = pyref.curve_point_from_x_search(C, 1000)
            assert C.on_curve(Q) and C.mul(C.r, Q) is not None
            h = (0xd201000000010000 + 1) ** 2 // 3                      # cofactor (z - 1)^2 / 3 with z = -0xd201000000010000
            assert C.mul(h * C.r, Q) is None
            small = C.mul(C.r * (h // (0xd201000000010000 + 1)), Q)     # order divides z - 1: the [x]P == P branch
            cleared = C.mul(h, Q)                                        # in the subgroup again
            for k, pt in ((7, Q), (8, small)):
                if pt is None:
                    continue
                bad = bytearray(good)
                bad[k * sz:(k + 1) * sz] = pyref.g1_serialize(C, [pt], compressed)
                assert both(bytes(bad), len(pts), compressed) == (k, pyref.WIRE_NOT_IN_SUBGROUP)
                assert both(bytes(bad), len(pts), compressed, validate=False) is None
            ok = bytearray(good)
            ok[7 * sz:8 * sz] = pyref.g1_serialize(C, [cleared], compressed)
            assert both(bytes(ok), len(pts), compressed) is None


def test_wire_kzg_containers(eng, pc):
    """Powers (two Vec<G1Affine>), Commitment and Proof framing around the element codec (kzg10/data_structures.rs:142-177,
    :315-328, :479-495): bytes equal the restated ark-serialize layout and read back to the same SRS."""
    import struct
    from poly_commit_b200 import wire
    cname = "bls12_381"
    C = pyref.Curve(cname)
    g = util.synthetic_srs(cname, 33, seed=5)
    gamma = util.random_points(cname, 3, seed=6)
    for compressed in (True, False):
        blob = wire.powers_serialize(eng, C.id, g, gamma, compressed)
        exp = (struct.pack("<Q", 33) + pyref.g1_serialize(C, C.points_from_limbs(g), compressed)
               + struct.pack("<Q", 3) + pyref.g1_serialize(C, C.points_from_limbs(gamma), compressed))
        assert blob == exp
        (g2, gi), (h2, hi) = wire.powers_deserialize(eng, C.id, blob, compressed)
        assert (g2 == g).all() and (h2 == gamma).all() and not gi.any() and not hi.any()
        with pytest.raises(ValueError):
            wire.powers_deserialize(eng, C.id, blob[:-1], compressed)
    # a commitment and a proof produced by the prover path
    srs = eng.srs_register(C.id, g)
    poly = util.rand_fr(cname, 33, seed=7, mont=True)
    comm, cinf = eng.kzg_commit(srs, poly)
    cb = wire.commitment_serialize(eng, C.id, comm, cinf)
    assert cb == pyref.g1_serialize(C, C.points_from_limbs(comm.reshape(1, -1), [cinf]), True)
    back, binf = wire.commitment_deserialize(eng, C.id, cb)
    assert (back == comm).all() and binf == bool(cinf)
    z = util.rand_fr(cname, 1, seed=8, mont=True)[0]
    w, winf, _ = eng.kzg_open(srs, poly, z)
    pb = wire.proof_serialize(eng, C.id, w, winf, None)
    assert pb == pyref.g1_serialize(C, C.points_from_limbs(w.reshape(1, -1), [winf]), True) + b"\x00"
    rv = util.rand_fr(cname, 1, seed=9, mont=True)[0]
    pb = wire.proof_serialize(eng, C.id, w, winf, rv)
    assert pb[-33] == 1 and int.from_bytes(pb[-32:], "little") == C.fr_from_limbs(rv, True)[0]


# ---- verifier-side combinations (SURVEY 8f rank 2) -------------------------------------------------------------------
@pytest.mark.parametrize("cname,n", [("bls12_381", 300), ("bn254", 65), ("pallas", 1)])
def test_msm_bases_unregistered(eng, pc, cname, n):
    """pcgpu_msm_bases == msm_bigint(bases, scalars) on fresh bases (hyrax/mod.rs:501-504), with an identity base and a
    zero scalar in the input; pcgpu_fr_mul == elementwise product."""
    C = pyref.Curve(cname)
    bases = util.random_points(cname, n, seed=80)
    inf = np.zeros(n, dtype=np.uint8)
    sc = util.rand_fr(cname, n, seed=81, mont=False)
    if n > 2:
        inf[1] = 1
        sc[2] = 0
    pts = C.points_from_limbs(bases, inf)
    exp = C.msm(pts, C.fr_from_limbs(sc, False))
    got, ginf = eng.msm_bases(C.id, bases, sc, inf=inf)
    ex, ei = C.points_to_limbs([exp])
    assert ginf == bool(ei[0]) and (got == ex[0]).all()
    a, b = util.rand_fr(cname, n, seed=82, mont=True), util.rand_fr(cname, n, seed=83, mont=True)
    prod = [x * y % C.r for x, y in zip(C.fr_from_limbs(a, True), C.fr_from_limbs(b, True))]
    assert (eng.fr_mul(C.id, a, b) == C.fr_to_limbs(prod, True)).all()


@pytest.mark.parametrize("hiding", [False, True])
def test_kzg10_batch_check_combination(eng, pc, hiding):
    """KZG10::batch_check's combination (kzg10/mod.rs:345-377) and check's inner point (:322-325) against the definition
    in Python integers, on REAL proofs from the prover path: the combined points must also satisfy the relation the pairing
    tests -- total_c = beta * (-neg_total_w) for the SRS's beta -- i.e. the batch verifies."""
    from poly_commit_b200 import kzg10
    cname = "bls12_381"
    C = pyref.Curve(cname)
    deg, m = 24, 5
    beta = C.fr_from_limbs(util.rand_fr(cname, 1, 1000 + 11, mont=True), True)[0]       # util.synthetic_srs's beta for seed 11
    g_pows = util.synthetic_srs(cname, deg + 1, seed=11)
    gamma_scalar = 0x1234567
    gamma_pts = [C.mul(gamma_scalar * pow(beta, i, C.r) % C.r, C.g) for i in range(3)]
    gamma_pows, _ = C.points_to_limbs(gamma_pts)
    srs, srs_gamma = eng.srs_register(C.id, g_pows), eng.srs_register(C.id, gamma_pows)
    comms, ws, zs, vs, rvs = [], [], [], [], []
    for k in range(m):
        poly = util.rand_fr(cname, deg + 1 - k, seed=90 + k, mont=True)
        blind = util.rand_fr(cname, 2, seed=95 + k, mont=True) if hiding else None
        z = util.rand_fr(cname, 1, seed=100 + k, mont=True)[0]
        if hiding:
            comm, cinf = eng.kzg_commit(srs, poly, powers_of_gamma_g=srs_gamma, blind=blind)
            w, winf, rv = eng.kzg_open(srs, poly, z, powers_of_gamma_g=srs_gamma, blind=blind)
            rvs.append(rv)
        else:
            comm, cinf = eng.kzg_commit(srs, poly)
            w, winf, _ = eng.kzg_open(srs, poly, z)
        assert not cinf and not winf
        comms.append(comm); ws.append(w); zs.append(z)
        vs.append(C.fr_to_limbs([pyref.poly_eval(C.fr_from_limbs(poly, True), C.fr_from_limbs(z, True)[0], C.r)], True)[0])
    rnd_int = [1] + [int(x) for x in util.rng(7).integers(1, 2**62, size=m - 1)]
    rnd_int = [x * x + 12345 for x in rnd_int]                                       # ~124-bit values, first one stays small
    rnd_int[0] = 1
    rnd = C.fr_to_limbs(rnd_int, True)
    g, gamma_g = g_pows[0], gamma_pows[0]
    (neg_w, nwinf), (tot_c, tcinf) = kzg10.batch_check_combine(eng, C.id, g, gamma_g, np.stack(comms), np.stack(zs), np.stack(vs),
                                                               np.stack(ws), rnd, np.stack(rvs) if hiding else None)
    # definition in Python integers
    cp, wp = C.points_from_limbs(np.stack(comms)), C.points_from_limbs(np.stack(ws))
    zi, vi = C.fr_from_limbs(np.stack(zs), True), C.fr_from_limbs(np.stack(vs), True)
    ri = C.fr_from_limbs(np.stack(rvs), True) if hiding else [0] * m
    tc, tw, gm, ggm = None, None, 0, 0
    for k in range(m):
        tc = C.add(tc, C.mul(rnd_int[k], C.add(cp[k], C.mul(zi[k], wp[k]))))
        tw = C.add(tw, C.mul(rnd_int[k], wp[k]))
        gm, ggm = (gm + rnd_int[k] * vi[k]) % C.r, (ggm + rnd_int[k] * ri[k]) % C.r
    tc = C.add(tc, C.neg(C.mul(gm, C.g)))
    tc = C.add(tc, C.neg(C.mul(ggm, gamma_pts[0])))
    ex, ei = C.points_to_limbs([C.neg(tw), tc])
    assert (neg_w == ex[0]).all() and (tot_c == ex[1]).all() and not nwinf and not tcinf
    # e(-total_w, beta h) * e(total_c, h) == 1  <=>  total_c == beta * total_w
    assert C.mul(beta, tw) == tc
    # single check: e(comm - g v - gamma_g rv, h) == e(w, beta h - z h)  <=>  inner == (beta - z) * w
    inner, iinf = kzg10.check_inner(eng, C.id, g, gamma_g, comms[0], vs[0], rvs[0] if hiding else None)
    exp_inner = C.mul((beta - zi[0]) % C.r, wp[0])
    ex, _ = C.points_to_limbs([exp_inner])
    assert (inner == ex[0]).all() and not iinf


# ---- Ligero row encoding (SURVEY 8f rank 4) --------------------------------------------------------------------------
def test_ligero_reed_solomon_like_the_reference(eng):
    """mirror of test_reed_solomon (linear_codes/utils.rs:303-331): rho_inv = 3, m = 2^i for i in 1..10 -- every encoded
    element equals the polynomial evaluated at the element of the larger domain."""
    from poly_commit_b200 import linear_codes
    cname = "bls12_381"
    C = pyref.Curve(cname)
    for i in range(1, 10):
        m = 1 << i
        coeffs = util.rand_fr(cname, m, seed=120 + i, mont=True)
        enc = linear_codes.reed_solomon(eng, C.id, coeffs, 3)
        logn = (3 * m - 1).bit_length()
        assert enc.shape[0] == 1 << logn
        w = C.domain_generator(logn)
        ci = C.fr_from_limbs(coeffs, True)
        for j in sorted({0, 1, 2, 3 * m - 1, (1 << logn) - 1, (7 * j0 + 3) % (3 * m) if (j0 := i) else 0}):
            assert C.fr_from_limbs(enc[j], True)[0] == pyref.poly_eval(ci, pow(w, j, C.r), C.r)
        assert (enc == orc.fr_ntt(C.id, coeffs, logn)).all()


def test_ligero_dimensions_like_the_reference():
    """test_calculate_t_with_good_parameters / _bad_parameters (linear_codes/utils.rs:344-360) on BLS12-377's 377-bit Fq"""
    from poly_commit_b200 import linear_codes
    assert linear_codes.calculate_t(377, 128, (3, 4), 2**32) < 200
    assert linear_codes.calculate_t(377, 256, (3, 4), 2**32) < 400
    with pytest.raises(ValueError):
        linear_codes.calculate_t(377, 377 - 60, (3, 4), 2**60)
    with pytest.raises(ValueError):
        linear_codes.calculate_t(377, 400, (3, 4), 2**32)
    n, m = linear_codes.compute_dimensions(0, 128, 4, 1 << 20)
    assert n & (n - 1) == 0 and n * m >= 1 << 20 and (m - 1) * n < 1 << 20


@pytest.mark.parametrize("cname,n_rows,n_cols,rho_inv,used", [("bls12_381", 8, 16, 4, 120), ("bn254", 3, 5, 2, 15),
                                                               ("pallas", 2, 1024, 4, 2048)])
def test_ligero_compute_matrices(eng, cname, n_rows, n_cols, rho_inv, used):
    """compute_matrices (linear_codes/mod.rs:118-138): row-major matrix, zero padding, every row through the NTT;
    the last case takes the four-step path (rows of 2^12)."""
    from poly_commit_b200 import linear_codes
    C = pyref.Curve(cname)
    coeffs = util.rand_fr(cname, used, seed=130, mont=True)
    mat, ext = linear_codes.compute_matrices(eng, C.id, coeffs, n_rows, n_cols, rho_inv)
    logn = (n_cols * rho_inv - 1).bit_length()
    assert ext.shape == (n_rows, 1 << logn, 4)
    flat = np.zeros((n_rows * n_cols, 4), dtype=np.uint64)
    flat[:used] = coeffs
    assert (mat.reshape(-1, 4) == flat).all() and (mat[1, 2] == flat[n_cols + 2]).all() if n_cols > 2 else True
    for r in range(n_rows):
        assert (ext[r] == orc.fr_ntt(C.id, flat[r * n_cols:(r + 1) * n_cols], logn)).all()
    # ifft of a row gives the row back (zero-padded)
    back = eng.ntt_batch(C.id, ext, logn, inverse=True)
    assert (back[:, :n_cols] == mat).all() and not back[:, n_cols:].any()


def test_msm_small_path_limits(eng, pc, monkeypatch):
    """csrc/msm_small.cuh at its edges: n = 4096 (largest one-launch size) and 4097 (first bucket-pipeline size) agree with
    the oracle; every digit value occurs (scalars built from all 64 six-bit patterns, incl. the -32 digit and the carry
    into the top window); the result does not depend on the path."""
    cname = "bn254"
    C = pyref.Curve(cname)
    bases = util.random_points(cname, 4097, seed=150)
    sc = util.rand_fr(cname, 4097, seed=151, mont=False)
    pats = []
    for d in range(64):
        v = sum(d << (6 * w) for w in range(43)) % C.r
        pats += [v, (C.r - 1 - v) % C.r]
    pats += [C.r - 1, C.r - 2, (1 << 253) - 1, 1 << 253, 32, 31, 33, (1 << 6) - 1]
    sc[:len(pats)] = C.fr_to_limbs(pats, False)
    srs = eng.srs_register(C.id, bases)
    for n in (4096, 4097, len(pats)):
        exp = orc.msm(C.id, bases, sc, n=n)
        got = eng.msm(srs, sc[:n], n=n)
        assert got[1] == exp[1] and (got[0] == exp[0]).all(), n
    monkeypatch.setenv("PCGPU_MSM_SMALL", "0")
    got = eng.msm(srs, sc[:len(pats)])
    assert (got[0] == orc.msm(C.id, bases, sc, n=len(pats))[0]).all()


@pytest.mark.parametrize("cname", ["bn254", "pallas"])
def test_glv_split_of_the_fold_challenge(hostcheck_path, cname):
    """host_glv.hpp: k = k1 + k2 * lambda (mod r) with both halves below 2^130, on edge and random scalars; lambda is the
    eigenvalue of phi(x, y) = (zeta x, y) on the generator (re-derived here in Python integers)."""
    lib = ctypes.CDLL(hostcheck_path)
    C = pyref.Curve(cname)
    r, p = C.r, C.p
    cands_l = [l for l in (pow(g, (r - 1) // 3, r) for g in range(2, 12)) if l != 1]
    cands_z = [z for z in (pow(g, (p - 1) // 3, p) for g in range(2, 12)) if z != 1]
    pairs = {(z, l) for z in cands_z for l in cands_l if C.mul(l, C.g) == (z * C.g[0] % p, C.g[1])}
    assert pairs
    lams = {l for _, l in pairs}
    g = np.random.default_rng(5)
    ks = [0, 1, 2, r - 1, r - 2, (r - 1) // 2, 1 << 128, (1 << 128) - 1, 1 << 254 if r > 1 << 254 else 1 << 253]
    ks += [int.from_bytes(g.bytes(32), "little") % r for _ in range(200)]
    used = None
    for k in ks:
        kin = np.array([(k >> (64 * j)) & (2**64 - 1) for j in range(4)], dtype=np.uint64)
        out = np.zeros(35, dtype=np.uint32)
        assert lib.hostcheck_glv(C.id, kin.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p)) == 0
        assert out[13] == 1, k
        # joint sparse form of (|k1|, |k2|) used by the fold kernel: digits in {-1, 0, 1} that reconstruct both magnitudes,
        # and of any two consecutive columns at most one is non-zero in the joint sense -- unless the pattern is the allowed
        # (+-1, 0), (+-1, +-1)-type pair of Solinas' form; the joint weight stays near one half of the columns
        ncols = int(out[14])
        mask = lambda base, j: (int(out[base + (j >> 5)]) >> (j & 31)) & 1  # noqa: E731
        u1 = [mask(15, j) * (-1 if mask(20, j) else 1) for j in range(ncols)]
        u2 = [mask(25, j) * (-1 if mask(30, j) else 1) for j in range(ncols)]
        m1 = sum(int(out[i]) << (32 * i) for i in range(5))
        m2 = sum(int(out[5 + i]) << (32 * i) for i in range(5))
        assert sum(d << j for j, d in enumerate(u1)) == m1 and sum(d << j for j, d in enumerate(u2)) == m2
        assert ncols <= int(out[12]) + 1
        if ncols > 100:
            weight = sum(1 for a, b in zip(u1, u2) if a or b)
            assert weight <= 0.62 * ncols, (weight, ncols)
        k1 = sum(int(out[i]) << (32 * i) for i in range(5)) * (-1 if out[10] else 1)
        k2 = sum(int(out[5 + i]) << (32 * i) for i in range(5)) * (-1 if out[11] else 1)
        assert abs(k1) < 1 << 130 and abs(k2) < 1 << 130 and out[12] == max(abs(k1).bit_length(), abs(k2).bit_length())
        ok = [l for l in lams if (k1 + k2 * l) % r == k]
        assert ok, k
        used = ok[0] if k > 2 else used
    assert used is not None


@pytest.mark.parametrize("cname,n", [("pallas", 16), ("bn254", 8)])
def test_ipa_fold_glv_equals_plain_ladder(eng, pc, cname, n, monkeypatch):
    """the GLV key fold (G1FoldGlvBody) and the 256-step ladder (G1FoldBody) give the same keys: identical l / r / final key
    with PCGPU_IPA_GLV=0 and =1, with an identity point in the key (the fold's early-out) and a tiny challenge."""
    from poly_commit_b200 import ipa_pc
    C = pyref.Curve(cname)
    key = util.random_points(cname, n, seed=170)
    key[n - 2] = 0                                               # identity in the right half
    h_prime = util.random_points(cname, 1, seed=171)[0]
    coeffs = util.rand_fr(cname, n, seed=172, mont=True)
    point = util.rand_fr(cname, 1, seed=173, mont=True)[0]
    outs = []
    for flag in ("1", "0"):
        monkeypatch.setenv("PCGPU_IPA_GLV", flag)
        outs.append(ipa_pc.open_rounds(eng, C.id, key, coeffs, point, h_prime, 3))
    for a, b in zip(outs[0]["l_vec"] + outs[0]["r_vec"], outs[1]["l_vec"] + outs[1]["r_vec"]):
        assert (a == b).all()
    assert (outs[0]["final_comm_key"] == outs[1]["final_comm_key"]).all()
    # and against the oracle on a key without the identity (the oracle's affine key has no encoding for it)
    key = util.random_points(cname, n, seed=174)
    monkeypatch.setenv("PCGPU_IPA_GLV", "1")
    got = ipa_pc.open_rounds(eng, C.id, key, coeffs, point, h_prime, 3)
    exp = oracle_ipa_rounds(cname, key, coeffs, point, h_prime, 3)
    assert (got["final_comm_key"] == exp["final_comm_key"]).all() and (got["c"] == exp["c"]).all()


def test_empty_inputs_on_the_widened_entry_points(eng, pc):
    """n = 0 everywhere: the identity / empty arrays, no error (msm_bigint of nothing is zero; an empty Vec serializes to its
    length prefix only)."""
    from poly_commit_b200 import wire
    cid = pc.BN254
    xy, inf = eng.msm_bases(cid, np.zeros((0, 8), dtype=np.uint64), np.zeros((0, 4), dtype=np.uint64))
    assert inf and not xy.any()
    assert eng.g1_serialize(cid, np.zeros((0, 8), dtype=np.uint64)).shape == (0, 32)
    assert eng.g1_deserialize(cid, b"", 0)[0].shape == (0, 8)
    assert eng.ntt_batch(cid, np.zeros((0, 4, 4), dtype=np.uint64), 3).shape == (0, 8, 4)
    blob = wire.powers_serialize(eng, cid, np.zeros((0, 8), dtype=np.uint64), np.zeros((0, 8), dtype=np.uint64))
    assert blob == bytes(16)
    (g, _), (h, _) = wire.powers_deserialize(eng, cid, blob)
    assert g.shape[0] == 0 and h.shape[0] == 0


@pytest.mark.parametrize("cname", ["bls12_381", "bn254", "pallas"])
@pytest.mark.parametrize("compressed", [True, False])
def test_wire_decode_fuzz_agrees_with_the_oracle(eng, pc, cname, compressed):
    """random byte strings, and valid encodings with single random bit flips: the device decoder and the Python restatement
    accept / reject the same inputs (same first offending index and reason) and decode accepted ones to the same points."""
    C = pyref.Curve(cname)
    sz = pyref.wire_size(C, compressed)
    g = np.random.default_rng(77 + sz)
    pts = C.points_from_limbs(util.random_points(cname, 6, seed=180))
    good = bytearray(pyref.g1_serialize(C, pts, compressed))
    cases = []
    for _ in range(60):                                   # bit flips in otherwise valid data
        b = bytearray(good)
        k = int(g.integers(0, len(b)))
        b[k] ^= 1 << int(g.integers(0, 8))
        cases.append(bytes(b))
    for _ in range(40):                                   # random blobs of 3 elements (flag bytes drawn from the interesting set)
        b = bytearray(g.integers(0, 256, size=3 * sz, dtype=np.uint8).tobytes())
        for e in range(3):
            pos = e * sz if cname == "bls12_381" else (e + 1) * sz - 1
            b[pos] = int(g.choice([0x00, 0x01, 0x20, 0x40, 0x80, 0x9f, 0xa0, 0xc0, 0xe0, 0x3f, 0x7f]))
        cases.append(bytes(b))
    accepted = 0
    for data in cases:
        n = len(data) // sz
        for validate in (True, False):
            try:
                exp, exp_err = pyref.g1_deserialize(C, data, n, compressed, validate), None
            except pyref.WireError as e:
                exp, exp_err = None, (e.index, e.reason)
            try:
                got, got_err = eng.g1_deserialize(C.id, data, n, compressed, validate), None
            except pc.binding.WireError as e:
                got, got_err = None, (e.index, e.reason)
            assert got_err == exp_err, (cname, compressed, validate, data.hex())
            if exp is not None:
                ex, ei = C.points_to_limbs(exp)
                assert (got[0] == ex).all() and (got[1] == ei).all()
                accepted += 1
    assert accepted > 0


@pytest.mark.parametrize("cname,n", [("bn254", 511), ("bn254", 512), ("pallas", 513), ("bls12_381", 1030)])
def test_msm_small_split_boundaries(eng, pc, cname, n):
    """the one-launch path around the size where a window's terms are divided among three blocks (512), with an identity
    base, repeated scalars and Montgomery input."""
    C = pyref.Curve(cname)
    bases = util.random_points(cname, n, seed=190)
    inf = np.zeros(n, dtype=np.uint8); inf[n // 2] = 1
    sc = util.rand_fr(cname, n, seed=191, mont=False)
    sc[10:40] = sc[10]
    sc[n - 1] = C.fr_to_limbs([C.r - 1], False)[0]
    srs = eng.srs_register(C.id, bases, inf=inf)
    exp = orc.msm(C.id, bases, sc, inf=inf)
    got = eng.msm(srs, sc)
    assert got[1] == exp[1] and (got[0] == exp[0]).all()
    scm = orc.field_unop("orc_fr_to_mont", C.id, sc)
    got = eng.msm(srs, scm, flags=pc.SCALARS_MONT)
    assert (got[0] == exp[0]).all()


@pytest.mark.parametrize("cname,which,fid", FIELDS)
def test_host_tail_field_product_vs_bigint(hostcheck_path, cname, which, fid):
    """host_ec.hpp's 64-bit Montgomery product (interleaved-carry CIOS, used by the MSM tail, to_affine and the GLV check) on
    edge values -- 0, 1, p-1, R, values with all-ones limbs -- and random ones, against Python integers."""
    lib = ctypes.CDLL(hostcheck_path)
    C = pyref.Curve(cname)
    mod = getattr(C, which)
    n64 = (mod.bit_length() + 63) // 64
    R = (1 << (64 * n64)) % mod
    Rinv = pow(R, -1, mod)
    g = np.random.default_rng(40 + fid)
    edge = [0, 1, 2, mod - 1, mod - 2, R, R * R % mod, mod >> 1, (mod >> 1) + 1, (1 << 64) - 1, ((1 << (64 * n64 - 2)) - 1) % mod,
            ((1 << (64 * (n64 - 1))) - 1), (mod - 1) ^ ((1 << 64) - 1) if mod > 1 << 64 else 3]
    edge = [e % mod for e in edge]
    rnd = [int.from_bytes(g.bytes(8 * n64), "little") % mod for _ in range(2000)]
    va = [a for a in edge for _ in edge] + rnd
    vb = [b for _ in edge for b in edge] + rnd[::-1]
    A, B = _tol(va, n64), _tol(vb, n64)
    out = np.zeros_like(A)
    vp = ctypes.c_void_p
    assert lib.hostcheck_hostfield_mul(fid, A.ctypes.data_as(vp), B.ctypes.data_as(vp), out.ctypes.data_as(vp), ctypes.c_size_t(len(va))) == 0
    assert (out == _tol([a * b * Rinv % mod for a, b in zip(va, vb)], n64)).all()


@pytest.mark.parametrize("cname,logn,world", [("bls12_381", 12, 2), ("bn254", 13, 4), ("pallas", 14, 8)])
def test_ntt_pass1_with_fused_exchange(eng, cname, logn, world):
    """pcgpu_ntt_pass1_peer: every "rank" transforms its columns and stores straight into the owners' row buffers (the fused
    all-to-all); pass 2 on each buffer then yields the same transform as the single call.  Ranks are simulated in-process:
    under emulation a device pointer is a host pointer, so the peer table is just the list of buffers."""
    C = pyref.Curve(cname)
    m1, m2 = eng.ntt_split(logn)
    N1, N2 = 1 << m1, 1 << m2
    rows, cols = N1 // world, N2 // world
    n_in = (1 << logn) - 5
    x = util.rand_fr(cname, n_in, seed=200 + logn, mont=True)
    for inverse in (False, True):
        rowbufs = [np.zeros((rows, N2, 4), dtype=np.uint64) for _ in range(world)]
        ptrs = [b.ctypes.data for b in rowbufs]
        for r in range(world):
            eng.ntt_pass1_peer(C.id, logn, r * cols, cols, x.ctypes.data, n_in, ptrs, inverse=inverse)
        outs = []
        for r in range(world):
            o = np.zeros((N2, rows, 4), dtype=np.uint64)
            eng.ntt_pass(C.id, logn, 2, r * rows, rows, rowbufs[r].ctypes.data, rows * N2, o.ctypes.data, inverse=inverse)
            outs.append(o)
        got = np.stack(outs, 0).transpose(1, 0, 2, 3).reshape(-1, 4)
        assert (got == eng.ntt(C.id, x, logn, inverse=inverse)).all()
    # the host-side driver (one engine per "device")
    from poly_commit_b200 import sharded
    pn = sharded.PeerNtt([eng] * world, C.id, logn)
    rowbufs = [np.zeros((rows, N2, 4), dtype=np.uint64) for _ in range(world)]
    outs = [np.zeros((N2, rows, 4), dtype=np.uint64) for _ in range(world)]
    pn.forward([x.ctypes.data] * world, n_in, [b.ctypes.data for b in rowbufs], [o.ctypes.data for o in outs])
    assert (np.stack(outs, 0).transpose(1, 0, 2, 3).reshape(-1, 4) == eng.ntt(C.id, x, logn)).all()
    with pytest.raises(Exception):
        eng.ntt_pass1_peer(C.id, logn, 0, cols, x.ctypes.data, n_in, [ptrs[0]] * 3)        # 3 ranks do not divide N1
    with pytest.raises(Exception):
        eng.ntt_pass1_peer(C.id, logn, N2 - 1, 2, x.ctypes.data, n_in, ptrs)                # columns out of range


def test_sonic_pc_host_mirror(eng, pc):
    """sonic_pc.commit / open (mirror of sonic_pc/mod.rs:274-382) vs the oracle composed the same way: a bounded polynomial is
    committed against shifted_powers(bound) only, and the opening is ONE KZG10 proof of the challenge-weighted combination."""
    from poly_commit_b200 import sonic_pc
    cname = "bls12_381"
    C = pyref.Curve(cname)
    max_degree, bounds = 40, [20, 33]
    pp = util.synthetic_srs(cname, max_degree + 1, seed=8)
    supported = 36
    powers = pp[: supported + 1]
    shifted = pp[max_degree - bounds[-1]:]                                   # trim(): powers_of_g[lowest_shift_degree..]
    ck = sonic_pc.CommitterKey(eng, C.id, powers, shifted, bounds)
    polys = [(util.rand_fr(cname, 30, seed=210, mont=True), None), (util.rand_fr(cname, 18, seed=211, mont=True), 20),
             (util.rand_fr(cname, 34, seed=212, mont=True), 33)]
    coms = sonic_pc.commit(ck, polys)
    for (coeffs, bound), comm in zip(polys, coms):
        key = powers if bound is None else shifted[bounds[-1] - bound:]
        rc, exy, einf = orc.kzg_commit(C.id, key, coeffs)
        assert rc == 0 and (comm[0] == exy).all() and comm[1] == einf
    # a bounded commitment is beta^(max_degree - bound) times the plain one: the relation the Sonic verifier's pairing checks
    beta = C.fr_from_limbs(util.rand_fr(cname, 1, 1000 + 8, mont=True), True)[0]
    plain = eng.kzg_commit(ck.powers, polys[1][0])
    shifted_pt = C.points_from_limbs(coms[1][0].reshape(1, -1))[0]
    assert C.mul(pow(beta, max_degree - 20, C.r), C.points_from_limbs(plain[0].reshape(1, -1))[0]) == shifted_pt
    point = util.rand_fr(cname, 1, seed=213, mont=True)[0]
    chals = util.rand_fr(cname, 3, seed=214, mont=True)
    w = sonic_pc.open(ck, polys, point, list(chals))
    p = np.zeros((34, 4), dtype=np.uint64)
    for (coeffs, _), c in zip(polys, chals):
        p[: len(coeffs)] = orc.fr_axpy(C.id, p[: len(coeffs)], c, coeffs)
    rc, w0, winf, _ = orc.kzg_open(C.id, powers, p, point)
    assert rc == 0 and (w[0] == w0).all() and w[1] == winf
    with pytest.raises(ValueError):
        sonic_pc.commit(ck, [(polys[2][0], 20)])                              # bound below the degree
    with pytest.raises(ValueError):
        sonic_pc.commit(ck, [(polys[1][0], 21)])                              # bound that was not enforced at trim


@pytest.mark.parametrize("cname", ["pallas", "bn254"])
def test_ipa_fold_special_challenges(eng, pc, cname, monkeypatch):
    """the key fold key_l + c * key_r (ipa_pc/mod.rs:699-701) for challenges that stress the GLV split -- 1, r-1, the
    eigenvalue lambda itself and its square (k1 = 0 or k2 = 0), powers of two around 2^128 -- with identity points in both
    halves: GLV ladder == 256-step ladder == the definition in Python integers."""
    from poly_commit_b200 import params
    C = pyref.Curve(cname)
    r = C.r
    lam = [l for l in (pow(g, (r - 1) // 3, r) for g in range(2, 12)) if l != 1][0]
    chals = [1, 2, r - 1, lam, lam * lam % r, (lam + 1) % r, 1 << 127, 1 << 128, (1 << 129) + 1, (r - 1) // 2, (lam << 64) % r]
    m = 4
    key = util.random_points(cname, 2 * m, seed=400)
    key[m + 1] = 0
    key[2] = 0
    inf = np.array([0 if k.any() else 1 for k in key], dtype=np.uint8)
    coeffs, z = util.rand_fr(cname, 2 * m, seed=1, mont=True), util.rand_fr(cname, 1, seed=2, mont=True)[0]
    for c in chals:
        outs = []
        for flag in ("1", "0"):
            monkeypatch.setenv("PCGPU_IPA_GLV", flag)
            st = eng.ipa_begin(C.id, key, coeffs, z)
            while eng.ipa_len(st) > 1:
                eng.ipa_round_fold(st, params.fr_mont(C.id, c), params.fr_mont(C.id, pow(c, -1, r)))
            outs.append(eng.ipa_finish(C.id, st)[0].copy())
        pts = C.points_from_limbs(key, inf=inf)
        while len(pts) > 1:
            h = len(pts) // 2
            pts = [C.add(pts[i], C.mul(c, pts[h + i])) for i in range(h)]
        ex, _ = C.points_to_limbs(pts)
        assert (outs[0] == outs[1]).all() and (outs[0].reshape(-1) == ex[0]).all(), hex(c)


@pytest.mark.parametrize("cname,n", [("pallas", 8192), ("bn254", 256)])
def test_ipa_frozen_key_rounds(eng, pc, cname, n, monkeypatch):
    """late rounds on a frozen key (csrc/ipa.cuh): explicit folds down to 4096 points, then weights instead of ladders.  Same
    l / r / final key / c as with explicit folds all the way (PCGPU_IPA_FREEZE=0), and the verifier's recomputed key matches."""
    from poly_commit_b200 import ipa_pc
    C = pyref.Curve(cname)
    key = util.random_points(cname, n, seed=270)
    h_prime = util.random_points(cname, 1, seed=271)[0]
    coeffs = util.rand_fr(cname, n - 5, seed=272, mont=True)
    point = util.rand_fr(cname, 1, seed=273, mont=True)[0]
    outs = []
    for flag in ("1", "0"):
        monkeypatch.setenv("PCGPU_IPA_FREEZE", flag)
        outs.append(ipa_pc.open_rounds(eng, C.id, key, coeffs, point, h_prime, 0x77))
    a, b = outs
    assert len(a["l_vec"]) == n.bit_length() - 1 and a["challenges"] == b["challenges"]
    for x, y in zip(a["l_vec"] + a["r_vec"], b["l_vec"] + b["r_vec"]):
        assert (x == y).all()
    assert (a["final_comm_key"] == b["final_comm_key"]).all() and (a["c"] == b["c"]).all()
    fk = ipa_pc.check_final_key(eng, C.id, key, a["challenges"])
    assert (fk[0] == a["final_comm_key"]).all()


@pytest.mark.parametrize("cname,name", [("pallas", b"PC-DL-2020"), ("bn254", b"Hyrax protocol"), ("bn254", b"PC-DL-2020")])
def test_sample_generators(eng, pc, cname, name):
    """InnerProductArgPC::sample_generators / HyraxPC::setup (ipa_pc/mod.rs:302-325, hyrax/mod.rs:143-163): hash-derived
    generators, including indices that need the retry counter and (BN254) digests whose flag bits select the smaller root"""
    C = pyref.Curve(cname)
    n = 64
    got = eng.g1_sample_generators(C.id, name, n, first_index=5)
    exp = pyref.sample_generators(C, name, n, first=5)
    assert C.points_from_limbs(got) == exp
    assert all(C.on_curve(P) for P in exp) and len(set(exp)) == n
    assert (eng.g1_sample_generators(C.id, name, 3, first_index=20) == got[15:18]).all()


@pytest.mark.parametrize("cname,logn,n_in,count", [("bls12_381", 12, 4000, 3), ("bn254", 13, 8192, 2), ("pallas", 12, 1, 2)])
def test_ntt_batch_long_rows(eng, cname, logn, n_in, count):
    """rows longer than one block pass (four-step per row): all rows' pass 1 in one launch, all rows' pass 2 in another ==
    one transform per row (forward and inverse)"""
    C = pyref.Curve(cname)
    rows = util.rand_fr(cname, count * n_in, seed=400 + logn, mont=True).reshape(count, n_in, 4)
    for inverse in (False, True):
        got = eng.ntt_batch(C.id, rows, logn, inverse=inverse)
        for r in range(count):
            assert (got[r] == eng.ntt(C.id, rows[r], logn, inverse=inverse)).all()
    assert (eng.ntt_batch(C.id, rows, logn)[0] == orc.fr_ntt(C.id, rows[0], logn)).all()
