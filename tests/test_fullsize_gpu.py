"""Parity at BASELINE.json's full block size (configs[1]: N = 100 000, bsize = 1000, P = 10; configs[2]: N = 500 000).

Direct comparison: one full block of each configuration against the compiled Eigen/OpenMP restatement of
calc_cv_matrices + ridge_level_0 (oracle/ref_eigen: the reference's own SelfAdjointEigenSolver, seconds per block),
1e-9 relative on every level-0 predictor column - the benchmarked k-fold path at the benchmarked size (16 Cholesky
panels, 72 Gram tiles, 5 prediction groups, folds of 20 000 / 100 000 samples).  The Eigen side is stored
(tests/golden/ref/, helpers.ref_golden): every column's max |W| and a fixed, seeded sample of 64 rows.

Size-independent identities on top (they hold for the reference's algorithm at any size):

  * level-0 predictors are centred and scaled per phenotype exactly as ridge_level_0 leaves them
    (src/Step1_Models.cpp:539-557):  sum_masked W = 0,  sum_masked W^2 = Neff - 1;
  * they are invariant to the scale and equivariant to the sign of the phenotype (the ridge solve is linear in Y,
    the standardisation removes the scale);
  * the same block under a different block id / stream lane gives bit-identical columns (fixed-order reductions);
  * Step-2 A1FREQ and N are exact functions of integer counts: compared bit for bit with a numpy popcount.
"""
import numpy as np
import pytest

import helpers
from regenie_b200 import hostprep, synth

pytestmark = pytest.mark.gpu

N, BS, P, C, K = 100_000, 1000, 10, 3, 5


@pytest.fixture(scope="module")
def panel():
    g = synth.genotypes(N, BS, seed=77, miss=0.01)
    Y, cov, na = synth.phenotypes(g, P, C, seed=78, n_causal=50, na_frac=0.02)
    X, Yr, mask, in_an, neff = hostprep.prepare_qt(Y, cov, na)
    return g, synth.pack_bed(g), X, Yr, mask, in_an, neff


def _step1(X, Y, mask, in_an, neff, total_blocks=3):
    from regenie_b200 import capi
    h0 = hostprep.ridge_grid(5)
    lam = 50_000 * (1 - h0) / h0
    return capi.Step1(X, Y, mask, in_an, hostprep.fold_sizes(N, K), lam, neff, N, BS, total_blocks)


def test_level0_full_block_matches_the_eigen_oracle_at_configs1(panel):
    """The benchmark configuration itself: N = 100k, bsize = 1000, 10 traits, 5 folds x 5 ridge values, 1 % missing
    calls, 2 % missing phenotypes - every one of the 50 predictor columns vs ridge_level_0 (src/Step1_Models.cpp:458-613)."""
    g, packed, X, Y, mask, in_an, neff = panel
    h0 = hostprep.ridge_grid(5)
    lam = 50_000 * (1 - h0) / h0
    fsz = hostprep.fold_sizes(N, K)

    def eigen():
        from oracle import ref_eigen
        return helpers.W_digest(ref_eigen.l0_block_kfold(packed, N, in_an, X, Y, mask, fsz, lam, neff, int(in_an.sum()))[0])
    W_o = helpers.ref_golden("level0_eigen_n100k", eigen)
    st = _step1(X, Y, mask, in_an, neff)
    st.l0_block_bed(packed, BS, 1)
    assert st.status() == 0
    W = [st.fetch_W(1, p) for p in range(P)]
    st.close()
    err = helpers.W_rel_err(W, W_o)
    assert err < 1e-9, "level-0 predictors at N=100k, bs=1000 differ from the Eigen oracle: %g" % err


def test_level0_full_block_properties(panel):
    g, packed, X, Y, mask, in_an, neff = panel
    st = _step1(X, Y, mask, in_an, neff)
    st.l0_block_bed(packed, BS, 0)
    st.l0_block_bed(packed, BS, 2)            # same rows again on another lane / block id
    assert st.status() == 0
    W0 = [st.fetch_W(0, p) for p in range(P)]
    for p in range(P):
        w = W0[p]
        assert np.isfinite(w).all()
        np.testing.assert_allclose(w.sum(axis=0), 0.0, atol=1e-6)                       # centred
        np.testing.assert_allclose((w * w).sum(axis=0), neff[p] - 1.0, rtol=1e-10)      # unit sd with the Neff - 1 divisor
        assert np.array_equal(w, st.fetch_W(2, p))                                      # bit-identical across lanes
    st.close()
    # scale invariance / sign equivariance in Y
    Y2 = np.asfortranarray(Y * np.array([3.0, -1.0, 0.25, -7.0, 1.0, 2.0, -2.0, 10.0, 0.5, -0.5])[None, :])
    st = _step1(X, Y2, mask, in_an, neff)
    st.l0_block_bed(packed, BS, 0)
    assert st.status() == 0
    sgn = np.sign([3.0, -1.0, 0.25, -7.0, 1.0, 2.0, -2.0, 10.0, 0.5, -0.5])
    for p in range(P):
        np.testing.assert_allclose(st.fetch_W(0, p), sgn[p] * W0[p], rtol=0, atol=2e-8)
    st.close()


def test_step2_counts_bit_exact_at_full_size(panel):
    from regenie_b200 import capi
    g, packed, X, Y, mask, in_an, neff = panel
    rng = np.random.default_rng(3)
    m2 = np.asfortranarray((rng.random((N, P)) > 0.03).astype(np.uint8))
    st = capi.Step2(X, m2, in_an, N, BS)
    st.set_chr(np.asfortranarray(Y * m2), np.ones(P))
    o = st.block_bed(packed)
    st.close()
    obs = g != 3
    gz = np.where(obs, g, 0).astype(np.int64)
    for p in range(P):
        mp = m2[:, p].astype(np.int64)
        ns = obs.astype(np.int64) @ mp
        tot = gz @ mp
        assert np.array_equal(o["ns"][:, p], ns)
        assert np.array_equal(o["af"][:, p], tot / (2.0 * ns))                           # bit for bit
    assert np.array_equal(o["ns_all"], obs.sum(axis=1))


def test_level0_block_at_n_500k():
    """BASELINE configs[2] sample count (N = 500 000, bsize = 1000, 10 traits): one block against the Eigen oracle
    (1e-9), plus the size-independent identities - standardisation sums, finite values, bit-identical columns when
    the block is replayed on another lane."""
    from regenie_b200 import capi
    n = 500_000
    rng = np.random.default_rng(123)
    maf = rng.uniform(0.01, 0.5, size=BS)
    g = rng.binomial(2, maf[:, None], size=(BS, n)).astype(np.uint8)
    g[rng.random(size=g.shape) < 0.01] = 3
    Y = rng.standard_normal((n, P))
    cov = rng.standard_normal((n, C - 1))
    X, Yr, mask, in_an, neff = hostprep.prepare_qt(Y, cov, None)
    h0 = hostprep.ridge_grid(5)
    packed = synth.pack_bed(g)

    def eigen():
        from oracle import ref_eigen
        return helpers.W_digest(ref_eigen.l0_block_kfold(packed, n, in_an, X, Yr, mask, hostprep.fold_sizes(n, K),
                                                         500_000 * (1 - h0) / h0, neff, int(in_an.sum()))[0])
    W_o = helpers.ref_golden("level0_eigen_n500k", eigen)
    st = capi.Step1(X, Yr, mask, in_an, hostprep.fold_sizes(n, K), 500_000 * (1 - h0) / h0, neff, n, BS, 2)
    st.l0_block_bed(packed, BS, 0)
    st.l0_block_bed(packed, BS, 1)
    assert st.status() == 0
    err = helpers.W_rel_err([st.fetch_W(0, p) for p in range(P)], W_o)
    assert err < 1e-9, "level-0 predictors at N=500k, bs=1000 differ from the Eigen oracle: %g" % err
    for p in (0, P - 1):
        w = st.fetch_W(0, p)
        assert np.isfinite(w).all()
        np.testing.assert_allclose(w.sum(axis=0), 0.0, atol=1e-5)
        np.testing.assert_allclose((w * w).sum(axis=0), neff[p] - 1.0, rtol=1e-10)
        assert np.array_equal(w, st.fetch_W(1, p))
    st.close()


def test_step2_counts_bit_exact_at_n_500k():
    """Step 2 at N = 500 000 (two sample chunks on the tensor-core path): N and A1FREQ bit for bit vs numpy counts, the
    test statistic against a direct float64 evaluation of compute_score_qt's dense formula for a few variants."""
    from regenie_b200 import capi
    n, m, p = 500_000, 256, 3
    rng = np.random.default_rng(77)
    maf = rng.uniform(0.02, 0.5, size=m)
    g = rng.binomial(2, maf[:, None], size=(m, n)).astype(np.uint8)
    g[rng.random(size=g.shape) < 0.01] = 3
    Y = rng.standard_normal((n, p))
    cov = rng.standard_normal((n, 2))
    X, Yr, mask, in_an, neff = hostprep.prepare_qt(Y, cov, None)
    m2 = np.asfortranarray((rng.random((n, p)) > 0.02).astype(np.uint8))
    res = np.asfortranarray(Yr * m2)
    st = capi.Step2(X, m2, in_an, n, m)
    st.set_chr(res, np.ones(p))
    o = st.block_bed(synth.pack_bed(g))
    st.close()
    obs = g != 3
    gz = np.where(obs, g, 0).astype(np.int64)
    for j in range(p):
        mp = m2[:, j].astype(np.int64)
        ns = obs.astype(np.int64) @ mp
        assert np.array_equal(o["ns"][:, j], ns)
        assert np.array_equal(o["af"][:, j], (gz @ mp) / (2.0 * ns))
    YtX = res.T @ X
    for i in (0, 100, 255):
        gi = np.where(obs[i], g[i], gz[i].sum() / obs[i].sum()).astype(np.float64)
        sparse = (gi != 0).sum() <= n * 0.5                        # check_sparse_G, src/Geno.cpp:3165
        assert bool(o["flags"][i] & 4) == sparse
        xtg = X.T @ gi
        gr = gi - X @ xtg
        for j in range(p):
            if sparse:                                             # src/Step2_Models.cpp:404, :410
                gm = gi * m2[:, j]
                num = res[:, j] @ gi - YtX[j] @ xtg
                den = gm @ gm - 2 * (X.T @ gm) @ xtg + xtg @ xtg
            else:                                                  # :415-416
                num = res[:, j] @ gr
                den = (m2[:, j] * gr * gr).sum()
            assert abs(o["stat"][i, j] - num / np.sqrt(den)) <= 1e-8 * max(1.0, abs(num / np.sqrt(den)))
