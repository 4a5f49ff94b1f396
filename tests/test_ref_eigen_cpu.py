"""The compiled Eigen/OpenMP restatement (oracle/ref_eigen, built against the reference's vendored Eigen 3.4.0) and
the numpy oracle are two independent restatements of the same reference functions; they must agree.  This gives the
QT k-fold level-0 arithmetic (which has no golden vector in the reference's tests, SURVEY 8c) a second pin that uses
the reference's own SelfAdjointEigenSolver, and the Step-2 QT score test a second implementation.  The Eigen side is
read from its stored outputs (tests/golden/ref/, helpers.ref_golden)."""
import numpy as np
import pytest

import helpers
from oracle import plink, step2


@pytest.mark.parametrize("seed,N,M,bsize", [(3, 1200, 160, 80), (11, 2051, 130, 130)])
def test_level0_kfold_eigen_matches_numpy_oracle(tmp_path, seed, N, M, bsize):
    pb = helpers.synthetic_problem(tmp_path, N=N, M=M, P=3, C=3, bsize=bsize, miss=0.02, seed=seed)
    pr = pb.prep

    def eigen():
        from oracle import ref_eigen
        out = {}
        for b in range(len(pb.blocks)):
            c, s, bs = pb.blocks[b]
            W_e, phases = ref_eigen.l0_block_kfold(pb.packed[s:s + bs], pb.n_file, pr.in_analysis, pr.X, pr.Y, pr.mask,
                                                   pb.fold_sizes, pb.lam, pr.neff, pr.n_analyzed, threads=2)
            assert (phases >= 0).all()
            out.update({"b%d_%s" % (b, k): v for k, v in helpers.W_digest(W_e).items()})
        return out
    ref = helpers.ref_golden("level0_kfold_eigen_seed%d" % seed, eigen)
    for b in range(len(pb.blocks)):
        W_np, _, _, _ = pb.oracle_l0(b)
        err = helpers.W_rel_err(W_np, ref, "b%d_" % b)
        assert err < 1e-9, (b, err)


def test_level0_eigen_is_thread_count_invariant_to_rounding(tmp_path):
    pb = helpers.synthetic_problem(tmp_path, N=900, M=64, P=2, C=3, bsize=64, seed=5)
    pr = pb.prep
    c, s, bs = pb.blocks[0]

    def eigen():
        from oracle import ref_eigen
        args = (pb.packed[s:s + bs], pb.n_file, pr.in_analysis, pr.X, pr.Y, pr.mask, pb.fold_sizes, pb.lam, pr.neff,
                pr.n_analyzed)
        out = {}
        for t in (1, 4):
            W, _ = ref_eigen.l0_block_kfold(*args, threads=t)
            out.update({"t%d_%s" % (t, k): v for k, v in helpers.W_digest(W).items()})
        return out
    ref = helpers.ref_golden("level0_eigen_threads", eigen)
    assert np.abs(ref["t1_W"] - ref["t4_W"]).max() < 1e-10
    assert np.abs(ref["t1_absmax"] - ref["t4_absmax"]).max() < 1e-10
    W_np, _, _, _ = pb.oracle_l0(0)
    for t in (1, 4):
        assert helpers.W_rel_err(W_np, ref, "t%d_" % t) < 1e-9


def test_step2_qt_eigen_matches_numpy_oracle(tmp_path):
    pb = helpers.synthetic_problem(tmp_path, N=1500, M=120, P=3, C=3, bsize=120, miss=0.03, seed=9)
    pr = pb.prep
    rng = np.random.default_rng(1)
    res = rng.normal(size=(pb.n_file, 3)) * pr.mask
    res /= np.linalg.norm(res, axis=0) / np.sqrt(pr.neff - pr.ncov)
    scf = np.array([1.3, 0.7, 2.0])
    YtX = res.T @ pr.X

    def eigen():
        from oracle import ref_eigen
        return {"out": ref_eigen.s2_block_qt_bed(pb.packed, pb.n_file, pr.in_analysis, pr.X, res, pr.mask, YtX, scf,
                                                 pr.n_analyzed, threads=2)}
    out = helpers.ref_golden("step2_qt_eigen", eigen)["out"]
    n_checked = 0
    for i in range(pb.M):
        graw = plink.decode_bed(pb.packed[i:i + 1], pb.n_file)[0]
        vs = step2.variant_stats(graw, pr.in_analysis, pr.mask)
        if vs["ignored"]:
            assert out[i, 0] == -1
            continue
        sc = step2.score_qt(vs["g"], pr.X, res, pr.mask, pr.in_analysis, pr.n_analyzed, pr.ncov, scf, YtX, False)
        assert out[i, 0] == vs["af1"] and out[i, 1] == vs["ns1"] and out[i, 3] == sc["is_sparse"]
        for ph in range(3):
            q = out[i, 4 + 5 * ph: 9 + 5 * ph]
            assert q[0] == vs["af"][ph] and q[1] == vs["ns"][ph]
            np.testing.assert_allclose(q[2:], [sc["beta"][ph], sc["se"][ph], sc["chisq"][ph]], rtol=1e-9)
        n_checked += 1
    assert n_checked > 50
