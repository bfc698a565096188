"""GPU parity tests (run with `-m gpu` on a B200): the CUDA library through its C ABI against the CPU oracle
on the same seeded inputs -- bit-exact (all arithmetic is integer / finite field; tolerance = 0).

Small and medium sizes compare directly against the oracle (definition-level MSM or its Pippenger); the
BASELINE.json size (2^20, BLS12-381) is compared directly as well (the C oracle's Pippenger finishes it in
seconds on the box's cores) and additionally through size-independent properties: linearity
(kzg10/mod.rs:520-544 add_commitments_test), index-range additivity, q*(X-z)+p(z) == p.
"""
import numpy as np
import pytest

from oracle import orc, pyref
from tests import util
# the same case bodies that run under host emulation, here against the real device
from tests.test_hostcheck import (test_fixed_base_mul, test_fr_div_linear, test_fr_vector_ops,  # noqa: F401
                                  test_kzg_commit_open, test_msm_edge_scalars, test_msm_infinity_bases,
                                  test_msm_partial_and_sum, test_msm_precomputed_tables, test_msm_vs_oracle,
                                  test_row_mul_reference_kat, test_golden_vectors, test_ntt_vs_oracle, test_msm_batch_shared_bases, test_ipa_open_rounds, test_msm_batched_affine_rounds, test_hyrax_host_mirror, test_marlin_pc_host_mirror, test_kzg_commit_batch, test_msm_two_level_reduction, test_msm_heavy_buckets,
                                  test_wire_roundtrip_vs_oracle, test_wire_bls12_381_generator_known_answer,
                                  test_wire_rejects_like_the_oracle, test_wire_kzg_containers, test_msm_bases_unregistered,
                                  test_kzg10_batch_check_combination, test_ligero_reed_solomon_like_the_reference, test_msm_small_path_limits, test_ipa_fold_glv_equals_plain_ladder, test_sonic_pc_host_mirror,
                                  test_ligero_compute_matrices, test_kzg_commit_open_fused, test_ipa_frozen_key_rounds, test_marlin_pc_hiding_and_bounds, test_sample_generators, test_ntt_batch_long_rows)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng(gpu_engine):
    return gpu_engine


def gpu_srs_beta(cname, seed=1):
    """the trapdoor beta (Montgomery form) of gpu_srs(..., seed): test_degenerate_srs checks commitments against p(beta) * G"""
    return util.rand_fr(cname, 1, 1000 + seed, mont=True)[0]


def gpu_srs(eng, cname, n, seed=1):
    """powers_of_g = beta^i * G built ON THE DEVICE (pcgpu_g1_fixed_base_mul), spot-checked against the oracle."""
    C = pyref.Curve(cname)
    beta = gpu_srs_beta(cname, seed)
    pows = orc.fr_powers_canonical(C.id, beta, n)
    xy = eng.fixed_base_mul(C.id, orc.g1_generator(C.id), pows)
    idx = np.unique(np.concatenate([[0, 1, n - 1], util.rng(seed).integers(0, n, size=12)]))
    exp, _ = orc.fixed_base_batch_mul(C.id, orc.g1_generator(C.id), pows[idx])
    assert (xy[idx] == exp).all()
    assert orc.g1_on_curve(C.id, xy[:: max(1, n // 4096)]) == 0
    return xy


@pytest.mark.parametrize("curve", [0, 1, 2])
def test_field_selftest(eng, curve):
    assert eng.selftest_field(curve, seed=3, n=1 << 16) == 0


@pytest.mark.parametrize("cname,logn", [("bls12_381", 10), ("bls12_381", 14), ("bls12_381", 16), ("bn254", 15), ("pallas", 15)])
def test_msm_medium(eng, pc, cname, logn):
    """cfg1 shape (2^10 + 1 coefficients) and medium sizes, raw bases and window-folded tables."""
    C = pyref.Curve(cname)
    n = (1 << logn) + 1
    bases = gpu_srs(eng, cname, n, seed=logn)
    sc = util.rand_fr(cname, n, seed=50 + logn, mont=False)
    exp = orc.msm(C.id, bases, sc)
    for flags in (0, pc.SRS_PRECOMPUTE):
        srs = eng.srs_register(C.id, bases, flags=flags)
        got = eng.msm(srs, sc)
        assert got[1] == exp[1] and (got[0] == exp[0]).all(), (cname, logn, flags)
        srs.release()


def test_msm_repeated_scalars_2p18(eng, pc):
    """2^18 coefficients of which 60 % are 1, -1 or 2 (heavy buckets of ~50 000 points in every window) plus 40 % uniform."""
    cname, n = "bls12_381", 1 << 18
    C = pyref.Curve(cname)
    bases = gpu_srs(eng, cname, n, seed=9)
    sc = util.rand_fr(cname, n, seed=62, mont=False)
    kind = util.rng(63).integers(0, 10, size=n)
    sc[kind < 2] = C.fr_to_limbs([1], False)[0]
    sc[(kind >= 2) & (kind < 4)] = C.fr_to_limbs([C.r - 1], False)[0]
    sc[(kind >= 4) & (kind < 6)] = C.fr_to_limbs([2], False)[0]
    exp = orc.msm(C.id, bases, sc)
    import time
    for flags in (0, pc.SRS_PRECOMPUTE):
        srs = eng.srs_register(C.id, bases, flags=flags)
        t0 = time.perf_counter()
        got = eng.msm(srs, sc)
        dt = time.perf_counter() - t0
        assert (got[0] == exp[0]).all()
        assert dt < 0.5, f"heavy-bucket MSM took {dt:.3f}s"
        srs.release()


def test_msm_skewed_scalars(eng, pc):
    """'witness-like' distribution (BASELINE.md): 50% zeros, 25% < 2^16, 25% uniform."""
    cname, n = "bls12_381", 1 << 15
    C = pyref.Curve(cname)
    bases = gpu_srs(eng, cname, n, seed=7)
    sc = util.rand_fr(cname, n, seed=60, mont=False)
    g = util.rng(61)
    kind = g.integers(0, 4, size=n)
    sc[kind < 2] = 0
    small = kind == 2
    sc[small, 1:] = 0
    sc[small, 0] &= np.uint64(0xFFFF)
    exp = orc.msm(C.id, bases, sc)
    for flags in (0, pc.SRS_PRECOMPUTE):
        srs = eng.srs_register(C.id, bases, flags=flags)
        got = eng.msm(srs, sc)
        assert (got[0] == exp[0]).all()
        srs.release()


@pytest.fixture(scope="module")
def big(eng, pc):
    """BASELINE.json cfg2 inputs: BLS12-381, 2^20 + 1 powers, a degree-2^20 polynomial."""
    cname = "bls12_381"
    C = pyref.Curve(cname)
    n = (1 << 20) + 1
    bases = gpu_srs(eng, cname, n, seed=20)
    coeffs = util.rand_fr(cname, n, seed=70, mont=True)
    srs = eng.srs_register(C.id, bases, flags=pc.SRS_PRECOMPUTE)
    raw = eng.srs_register(C.id, bases)
    return dict(C=C, n=n, bases=bases, coeffs=coeffs, srs=srs, raw=raw)


def test_cfg2_commit_open_vs_oracle(eng, big):
    """MarlinKZG10 commit+open, degree 2^20, BLS12-381: bit-exact against the C oracle (both MSM paths)."""
    C, n = big["C"], big["n"]
    z = util.rand_fr("bls12_381", 1, seed=71, mont=True)[0]
    rc, exy, einf = orc.kzg_commit(C.id, big["bases"], big["coeffs"])
    assert rc == 0
    for srs in (big["srs"], big["raw"]):
        got = eng.kzg_commit(srs, big["coeffs"])
        assert got[1] == einf and (got[0] == exy).all()
    rc, wxy, winf, _ = orc.kzg_open(C.id, big["bases"], big["coeffs"], z)
    assert rc == 0
    got = eng.kzg_open(big["srs"], big["coeffs"], z)
    assert got[1] == winf and (got[0] == wxy).all()


def test_cfg2_fused_commit_open(eng, pc, big):
    """the one-call commit+open (two overlapped MSM pipelines, one upload) at the cfg2 size, host and device-resident inputs"""
    import torch
    C, n = big["C"], big["n"]
    z = util.rand_fr("bls12_381", 1, seed=71, mont=True)[0]
    rc, exy, einf = orc.kzg_commit(C.id, big["bases"], big["coeffs"])
    rc2, wxy, winf, _ = orc.kzg_open(C.id, big["bases"], big["coeffs"], z)
    assert rc == 0 and rc2 == 0
    (c, ci), (w, wi) = eng.kzg_commit_open(big["srs"], big["coeffs"], z)
    assert (c == exy).all() and ci == einf and (w == wxy).all() and wi == winf
    # three distinct polynomials in flight: a result in the wrong slot or cross-talk between the ways shows.  The two new ones are
    # checked against the trapdoor formulas (p(beta) * G, test_degenerate_srs), the first against the oracle above.
    from tests.test_degenerate_srs import ref_commit, ref_witness
    beta = C.fr_from_limbs(gpu_srs_beta("bls12_381", 20), True)[0]
    zi = C.fr_from_limbs(z, True)[0]
    others = [util.rand_fr_fast("bls12_381", n, seed=75), util.rand_fr_fast("bls12_381", n // 2 + 3, seed=76)]
    others[0][-4321:] = 0
    exp = [((exy, einf), (wxy, winf))] + [(ref_commit(C, p, beta), ref_witness(C, p, beta, zi)) for p in others]
    ds = [torch.from_numpy(p.view(np.int64)).cuda() for p in [big["coeffs"]] + others]
    cb, cib, wb, wib = eng.kzg_commit_open_batch(big["srs"], [(d.data_ptr(), d.shape[0]) for d in ds], z, flags=pc.DEVICE_PTRS)
    for i, ((ec, eci), (ew, ewi)) in enumerate(exp):
        assert cib[i] == eci and wib[i] == ewi and (cb[i] == ec).all() and (wb[i] == ew).all(), i


def test_cfg2_properties(eng, pc, big):
    """size-independent properties at 2^20: linearity, index-range additivity, division identity."""
    C, n = big["C"], big["n"]
    srs = big["srs"]
    p = big["coeffs"]
    f = util.rand_fr("bls12_381", 1, seed=72, mont=True)[0]
    # commit(f * p) == f * commit(p)     (add_commitments_test, kzg10/mod.rs:520-544)
    fp = eng.fr_axpy(C.id, np.zeros_like(p), f, p)
    c1 = eng.kzg_commit(srs, fp)
    c0 = eng.kzg_commit(srs, p)
    f_canon = orc.field_unop("orc_fr_from_mont", C.id, f.reshape(1, 4))
    exp, _ = orc.g1_mul(C.id, c0[0], f_canon)
    assert (c1[0] == exp).all()
    # sum of index-range partials == whole
    cuts = [0, n // 3, n // 2, n]
    parts = [eng.msm_partial(srs, p[a:b], n=b - a, base_offset=a, flags=pc.SCALARS_MONT) for a, b in zip(cuts[:-1], cuts[1:])]
    tot = eng.g1_sum_xyzz(C.id, np.concatenate(parts))
    assert (tot[0] == c0[0]).all()
    # division: q*(X - z) + rem == p, checked at a second random point t:  q(t)*(t - z) + rem == p(t)
    z = util.rand_fr("bls12_381", 1, seed=73, mont=True)[0]
    t = util.rand_fr("bls12_381", 1, seed=74, mont=True)[0]
    q, rem = eng.fr_div_linear(C.id, p, z)
    _, qt = eng.fr_div_linear(C.id, q, t)
    _, pt = eng.fr_div_linear(C.id, p, t)
    zi, ti, qi, ri, pi = (C.fr_from_limbs(a, True)[0] for a in (z, t, qt, rem, pt))
    assert (qi * (ti - zi) + ri) % C.r == pi
    assert (rem == orc.fr_eval(C.id, p, z)).all()


def test_device_pointer_path(eng, pc, big):
    """PCGPU_DEVICE_PTRS: scalars already resident in HBM (the bench's `value` leg) give the same point."""
    import torch
    C, n = big["C"], big["n"]
    p = big["coeffs"]
    d = torch.from_numpy(p.view(np.int64)).cuda()
    got = eng.kzg_commit(big["srs"], d.data_ptr(), n=n, flags=pc.DEVICE_PTRS)
    exp = eng.kzg_commit(big["srs"], p)
    assert (got[0] == exp[0]).all()


@pytest.mark.parametrize("cname,logn", [("bls12_381", 20), ("bn254", 18), ("pallas", 21)])
def test_ntt_large(eng, cname, logn):
    """north_star size (2^20, BLS12-381 Fr): bit-exact vs the oracle's recursive NTT, and ifft(fft(x)) == x."""
    C = pyref.Curve(cname)
    n_in = (1 << logn) - 12345
    x = util.rand_fr_fast(cname, n_in, seed=400 + logn)
    got = eng.ntt(C.id, x, logn)
    assert (got == orc.fr_ntt(C.id, x, logn)).all()
    back = eng.ntt(C.id, got, logn, inverse=True)
    assert (back[:n_in] == x).all() and not back[n_in:].any()


@pytest.mark.parametrize("cname,logn,world", [("bls12_381", 20, 4), ("bn254", 14, 2)])
def test_ntt_passes_sharded_on_one_gpu(eng, cname, logn, world):
    """pcgpu_ntt_pass (the building block of sharded.ShardedNtt, SURVEY 8e): run every rank's slice of both passes on one
    device, do the all-to-all as a tensor permutation, and compare with the single-call transform."""
    import torch
    C = pyref.Curve(cname)
    m1, m2 = eng.ntt_split(logn)
    N1, N2 = 1 << m1, 1 << m2
    cols, rows = N2 // world, N1 // world
    n_in = (1 << logn) - 77
    x = util.rand_fr_fast(cname, n_in, seed=410 + logn)
    dev = torch.device("cuda", 0)
    xd = torch.from_numpy(x.view(np.int64).copy()).to(dev)
    a = [torch.empty((N1, cols, 4), dtype=torch.int64, device=dev) for _ in range(world)]
    torch.cuda.synchronize()
    for r in range(world):
        eng.ntt_pass(C.id, logn, 1, r * cols, cols, xd.data_ptr(), n_in, a[r].data_ptr())
    outs = []
    for r in range(world):
        rowbuf = torch.cat([a[s][r * rows:(r + 1) * rows] for s in range(world)], dim=1).contiguous()   # [k1_local][n2]
        o = torch.empty((N2, rows, 4), dtype=torch.int64, device=dev)
        torch.cuda.synchronize()
        eng.ntt_pass(C.id, logn, 2, r * rows, rows, rowbuf.data_ptr(), rows * N2, o.data_ptr())
        outs.append(o)
    got = torch.stack(outs, 0).permute(1, 0, 2, 3).contiguous().reshape(-1, 4).cpu().numpy().view(np.uint64)
    assert (got == eng.ntt(C.id, x, logn)).all()
    with pytest.raises(Exception):
        eng.ntt_pass(C.id, logn, 1, N2 - 1, 2, xd.data_ptr(), n_in, a[0].data_ptr())


@pytest.mark.parametrize("cname,logn", [("bls12_381", 18), ("pallas", 16)])
def test_wire_srs_ingest_large(eng, pc, cname, logn):
    """SRS ingestion at size (SURVEY 8f rank 1): serialize 2^k powers, read them back compressed with validation
    (square root + subgroup check per point on the device) and uncompressed; sampled elements against the Python
    restatement; a corrupted element deep in the file is located exactly."""
    C = pyref.Curve(cname)
    n = 1 << logn
    g = gpu_srs(eng, cname, n, seed=70)
    for compressed in (True, False):
        blob = eng.g1_serialize(C.id, g, None, compressed)
        idx = np.unique(np.concatenate([[0, 1, n - 1], util.rng(71).integers(0, n, size=40)]))
        assert blob[idx].tobytes() == pyref.g1_serialize(C, C.points_from_limbs(g[idx]), compressed)
        back, inf = eng.g1_deserialize(C.id, blob, n, compressed, validate=True)
        assert (back == g).all() and not inf.any()
    bad = blob.copy()
    k = n - 12345
    bad[k, 3] ^= 0x55                                           # uncompressed y no longer matches x
    with pytest.raises(pc.binding.WireError) as ei:
        eng.g1_deserialize(C.id, bad, n, False, validate=True)
    assert ei.value.index == k and ei.value.reason in (pyref.WIRE_NOT_ON_CURVE, pyref.WIRE_NOT_CANONICAL)


def test_ligero_rows_at_size(eng):
    """Ligero matrix for a 2^20-coefficient polynomial: 1024 rows of 1024 coefficients encoded at rate 1/2 (2^11-point rows) in ONE launch;
    sampled rows against the oracle, all rows through decode(encode(row)) == row."""
    cname = "bls12_381"
    C = pyref.Curve(cname)
    n_rows, n_cols, logn = 1024, 1024, 12 - 1
    mat = util.rand_fr_fast(cname, n_rows * n_cols, seed=140).reshape(n_rows, n_cols, 4)
    ext = eng.ntt_batch(C.id, mat, logn)
    for r in (0, 1, 511, 1023):
        assert (ext[r] == orc.fr_ntt(C.id, mat[r], logn)).all()
    back = eng.ntt_batch(C.id, ext, logn, inverse=True)
    assert (back[:, :n_cols] == mat).all() and not back[:, n_cols:].any()


def test_cfg4_hyrax_commit_rows(eng, pc):
    """BASELINE.json cfg4: Hyrax, 22 variables, BN254 -- 2^11 Pedersen row commitments over one com_key (+ h * r_i)
    (hyrax/mod.rs:233-242).  Row randomness is an INPUT (the reference draws it from thread_rng, :237-238, so parity is
    asserted at pedersen_commit level).  Checks: sampled rows vs one oracle MSM each; the sum of all row commitments vs
    the oracle MSM of the column sums (linearity over the whole matrix)."""
    cname = "bn254"
    C = pyref.Curve(cname)
    dim = 1 << 11
    bases = gpu_srs(eng, cname, dim + 1, seed=30)                 # com_key || h  (synthetic generators k_i * G)
    mat = util.rand_fr_fast(cname, dim * (dim + 1), seed=31).reshape(dim, dim + 1, 4)   # evaluations || r_i
    srs = eng.srs_register(C.id, bases, flags=pc.SRS_COMB)
    got, inf = eng.msm_batch(srs, mat, dim + 1, dim, flags=pc.SCALARS_MONT)
    assert not inf.any()
    for r in (0, 1, 777, dim - 1):
        exp = orc.msm(C.id, bases, orc.field_unop("orc_fr_from_mont", C.id, mat[r]))
        assert (got[r] == exp[0]).all(), r
    ones = np.tile(util.fr_const(cname, 1), (dim, 1))
    colsum = eng.fr_row_mul(C.id, ones, mat.reshape(-1, 4), dim, dim + 1)
    exp = orc.msm(C.id, bases, orc.field_unop("orc_fr_from_mont", C.id, colsum))
    tot = orc.g1_sum(C.id, got)
    assert (tot[0] == exp[0]).all()
    # Hyrax open's matrix-vector product (hyrax/mod.rs:347 -> utils.rs:127-146) at full size, sampled columns vs oracle
    l = util.rand_fr_fast(cname, dim, seed=32)
    lt = eng.fr_row_mul(C.id, l, mat.reshape(-1, 4), dim, dim + 1)
    for cidx in (0, 5, dim):
        col = np.ascontiguousarray(mat[:, cidx, :])
        assert (lt[cidx] == orc.fr_inner_product(C.id, l, col)).all()


def test_cfg3_ipa_open_2p18_pallas(eng, pc):
    """BASELINE.json cfg3: InnerProductArgPC open, degree 2^18 - 1, Pallas: the whole 18-round loop on the device;
    parity through (i) round-1 l and r against the oracle directly, (ii) the closed forms of the loop:
    c = sum_i coeffs[i] * prod_j inv_j^{b_j(i)},  final_comm_key = sum_i (prod_j chal_j^{b_j(i)}) key[i]."""
    from poly_commit_b200 import ipa_pc
    cname = "pallas"
    C = pyref.Curve(cname)
    logn = 18
    n = 1 << logn
    key = gpu_srs(eng, cname, n, seed=40)
    h_prime = util.random_points(cname, 1, seed=41)[0]
    coeffs = util.rand_fr_fast(cname, n, seed=42)
    point = util.rand_fr(cname, 1, seed=43, mont=True)[0]
    got = ipa_pc.open_rounds(eng, C.id, key, coeffs, point, h_prime, 0xabcdef)
    assert len(got["l_vec"]) == logn
    # (i) first round against the oracle
    m = n // 2
    z_int = C.fr_from_limbs(point, True)[0]
    co_int = C.fr_from_limbs(coeffs, True)
    zp = [1] * n
    for i in range(1, n):
        zp[i] = zp[i - 1] * z_int % C.r
    def cm(keypart, sc_ints, ip):
        msm, inf = orc.msm(C.id, keypart, C.fr_to_limbs(sc_ints, False))
        hp, hinf = orc.g1_mul(C.id, h_prime, C.fr_to_limbs([ip], False))
        return orc.g1_sum(C.id, np.stack([msm, hp]), inf=np.array([inf, hinf], dtype=np.uint8))[0]
    l0 = cm(key[:m], co_int[m:], sum(a * b for a, b in zip(co_int[m:], zp[:m])) % C.r)
    r0 = cm(key[m:], co_int[:m], sum(a * b for a, b in zip(co_int[:m], zp[m:])) % C.r)
    assert (got["l_vec"][0] == l0).all() and (got["r_vec"][0] == r0).all()
    # (ii) closed forms
    ch = got["challenges"]
    inv = [pow(c, -1, C.r) for c in ch]
    s_ch, s_inv = [1], [1]
    for j in range(logn - 1, -1, -1):          # last round pairs neighbours (lowest bit), first round the top bit
        s_ch = s_ch + [x * ch[j] % C.r for x in s_ch]
        s_inv = s_inv + [x * inv[j] % C.r for x in s_inv]
    c_exp = sum(a * b for a, b in zip(co_int, s_inv)) % C.r
    assert C.fr_from_limbs(got["c"], True)[0] == c_exp
    fk = orc.msm(C.id, key, C.fr_to_limbs(s_ch, False))
    assert (got["final_comm_key"] == fk[0]).all()
    # the verifier's linear-time step on the device (check_poly.compute_coeffs() + cm_commit, ipa_pc/mod.rs:760-766)
    vk = ipa_pc.check_final_key(eng, C.id, key, ch)
    assert (vk[0] == got["final_comm_key"]).all()


def test_cpp_host_mirror(tmp_path):
    """poly-commit_b200/host/pcgpu.hpp (C++ mirror of kzg10::KZG10::{commit, open}, Powers, Error) driven by the compiled
    tests/cpp/host_mirror_test -- the shape of kzg10/mod.rs:546-575 end_to_end_test_template -- against the oracle."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "tests", "cpp", "host_mirror_test")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-s", "-C", os.path.join(root, "tests", "cpp")])
    cname = "bls12_381"
    C = pyref.Curve(cname)
    n = 5000
    powers = util.synthetic_srs(cname, 512, seed=3)
    powers = np.concatenate([powers] + [util.random_points(cname, n - 512, seed=4)])
    gammas = util.random_points(cname, 6, seed=5)
    coeffs = util.rand_fr(cname, n - 7, seed=6, mont=True)
    blind = util.rand_fr(cname, 3, seed=7, mont=True)
    z = util.rand_fr(cname, 1, seed=8, mont=True)[0]
    fin, fout = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(fin, "wb") as f:
        f.write(np.array([C.id, n, n - 7, 6, 3], dtype=np.uint32).tobytes())
        for a in (powers, coeffs, z, gammas, blind):
            f.write(np.ascontiguousarray(a, dtype=np.uint64).tobytes())
    subprocess.check_call([exe, str(fin), str(fout)])
    raw = open(fout, "rb").read()
    pts = np.frombuffer(raw[: 4 * 96], dtype=np.uint64).reshape(4, 12)
    rv = np.frombuffer(raw[4 * 96: 4 * 96 + 32], dtype=np.uint64)
    kind = int(np.frombuffer(raw[4 * 96 + 32:], dtype=np.uint32)[0])
    rc, c0, _ = orc.kzg_commit(C.id, powers, coeffs)
    rc, w0, _, _ = orc.kzg_open(C.id, powers, coeffs, z)
    rc, c1, _ = orc.kzg_commit(C.id, powers, coeffs, gammas, blind)
    rc, w1, _, erv = orc.kzg_open(C.id, powers, coeffs, z, gammas, blind)
    assert (pts[0] == c0).all() and (pts[1] == w0).all() and (pts[2] == c1).all() and (pts[3] == w1).all()
    assert (rv == erv).all()
    assert kind == 0  # Error::TooManyCoefficients


def test_cfg5_shape_2p22(eng, pc):
    """BASELINE.json cfg5's per-polynomial shape (degree 2^22, BLS12-381; the 64-polynomial batch is 64 such commits
    spread over the GPUs, poly_assignment): one commit against the oracle directly, plus linearity between two
    polynomials:  commit(p0 + f*p1) == commit(p0) + f*commit(p1)."""
    cname = "bls12_381"
    C = pyref.Curve(cname)
    n = (1 << 22) + 1
    bases = gpu_srs(eng, cname, n, seed=50)
    srs = eng.srs_register(C.id, bases, flags=pc.SRS_PRECOMPUTE)
    p0 = util.rand_fr_fast(cname, n, seed=500)
    p1 = util.rand_fr_fast(cname, n, seed=501)
    c0 = eng.kzg_commit(srs, p0)
    c1 = eng.kzg_commit(srs, p1)
    rc, e0, _ = orc.kzg_commit(C.id, bases, p0)
    assert rc == 0 and (c0[0] == e0).all()
    f = util.rand_fr(cname, 1, seed=502, mont=True)[0]
    comb = eng.fr_axpy(C.id, p0, f, p1)
    cc = eng.kzg_commit(srs, comb)
    fc1, _ = orc.g1_mul(C.id, c1[0], orc.field_unop("orc_fr_from_mont", C.id, f.reshape(1, 4)))
    exp, _ = orc.g1_sum(C.id, np.stack([c0[0], fc1]))
    assert (cc[0] == exp).all()
    # the batch entry point (4 polynomials in flight on sibling contexts) returns the same commitments
    got, inf = eng.kzg_commit_batch(srs, [p0, p1, comb, p0, p1])
    assert (got[0] == c0[0]).all() and (got[1] == c1[0]).all() and (got[2] == cc[0]).all() and (got[3] == c0[0]).all()
    assert not inf.any()
    srs.release()


@pytest.mark.parametrize("cname,logn", [("bls12_381", 22), ("pallas", 19)])
def test_div_linear_one_pass_equals_level_tree(eng, cname, logn, monkeypatch):
    """The one-pass division (tiles chained by a decoupled look-back: at 2^22 the first wave of ~450 resident tiles walks several
    look-back windows over aggregate-only predecessors) against the level tree, bit for bit, and against p(z) from the oracle."""
    C = pyref.Curve(cname)
    n = (1 << logn) + 77
    p = util.rand_fr_fast(cname, n, seed=400 + logn)
    z = util.rand_fr(cname, 1, seed=401, mont=True)[0]
    monkeypatch.setenv("PCGPU_DIV_MODE", "tile")
    q1, r1 = eng.fr_div_linear(C.id, p, z)
    for _ in range(3):      # the look-back's timing differs from run to run: repeat
        q1b, r1b = eng.fr_div_linear(C.id, p, z)
        assert (q1b == q1).all() and (r1b == r1).all()
    monkeypatch.setenv("PCGPU_DIV_MODE", "tree")
    q2, r2 = eng.fr_div_linear(C.id, p, z)
    assert (q1 == q2).all() and (r1 == r2).all()
    assert (r1 == orc.fr_eval(C.id, p, z)).all()


def test_concurrent_host_threads(eng, pc):
    """Re-entrancy (SURVEY 8b): HyraxPC::commit calls msm from inside a Rayon par_iter (hyrax/mod.rs:233-242).  Eight host
    threads -- four sharing ONE context (calls serialised by its mutex), four with a context each -- run MSMs of different
    scalar vectors over one registered SRS at the same time; every result equals the oracle's."""
    import threading
    cname = "bn254"
    C = pyref.Curve(cname)
    n = (1 << 14) + 3
    bases = gpu_srs(eng, cname, n, seed=77)
    srs = eng.srs_register(C.id, bases, flags=pc.SRS_PRECOMPUTE)
    scalars = [util.rand_fr(cname, n, seed=900 + t, mont=False) for t in range(8)]
    expected = [orc.msm(C.id, bases, s) for s in scalars]
    own = [pc.Engine(0) for _ in range(4)]
    engines = [eng] * 4 + own
    got, errors = [None] * 8, []

    def work(t):
        try:
            for _ in range(6):
                got[t] = engines[t].msm(srs, scalars[t])
        except Exception as e:  # noqa: BLE001
            errors.append((t, repr(e)))

    threads = [threading.Thread(target=work, args=(t,)) for t in range(8)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    for e in own:
        e.close()
    assert not errors, errors
    for t in range(8):
        assert (got[t][0] == expected[t][0]).all() and got[t][1] == expected[t][1], f"thread {t}"


def test_randomised_sweep(capsys):
    """A short run of tests/perf/fuzz_gpu.py (random shapes across the small-path / split / bucket-pipeline boundaries, scalar
    mixtures, base offsets, the three division modes, NTT + inverse, hiding commits / opens), bit-exact against the C oracle;
    profiles/r02_fuzz_gpu.log holds two 400-case runs."""
    import importlib.util
    import os
    import sys
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "perf", "fuzz_gpu.py")
    spec = importlib.util.spec_from_file_location("fuzz_gpu", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    argv = sys.argv
    try:
        sys.argv = [path, "80", "4242"]
        mod.main()
    finally:
        sys.argv = argv
    assert '"ok": true' in capsys.readouterr().out
