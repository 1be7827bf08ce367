"""CPU: the VBx oracle against the outputs of the reference's own VBx.py and the golden fixture;
the host restatement of scipy's maxclust flat clustering against scipy."""
import os

import numpy as np
import pytest

from oracle import vbx_oracle
import vbx_util

GOLD = os.path.join(os.path.dirname(__file__), "golden", "vbx.npz")
PINS = os.path.join(os.path.dirname(__file__), "golden", "reference_pins.npz")


def _case(seed=0):
    xt, plda = vbx_util.make_plda(seed)
    emb, seg = vbx_util.make_embeddings(seed)
    return xt, plda, emb, seg


def test_vb_gmm_matches_golden():
    g = np.load(GOLD)
    gamma, pi, hist = vbx_oracle.vb_gmm(g["fea"], g["phi"], g["q0"], float(g["Fa"]), float(g["Fb"]), int(g["max_iters"]))
    np.testing.assert_allclose(gamma, g["gamma"], rtol=0, atol=1e-10)
    np.testing.assert_allclose(pi, g["pi"], rtol=0, atol=1e-12)


def test_plda_setup_matches_golden():
    g = np.load(GOLD)
    xt, plda = vbx_util.make_plda(int(g["seed"]))
    xvec_tf, plda_tf, psi = vbx_oracle.plda_setup(xt, plda)
    np.testing.assert_allclose(psi, g["psi"], rtol=1e-10)
    fea = plda_tf(xvec_tf(g["train"]), lda_dim=g["fea"].shape[1])
    # generalized eigenvectors are defined up to sign
    np.testing.assert_allclose(np.abs(fea), np.abs(g["fea"]), rtol=0, atol=1e-8)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_equals_reference_vbx(seed):
    """against the reference's vbx_setup (PLDA written as vbx_util.write_plda does) and cluster_vbx on the same labels
    (their outputs: reference_pins.npz)"""
    z = np.load(PINS)
    xt, plda, emb, seg = _case(seed)
    from oracle.pipeline_oracle import filter_embeddings
    train, _, _ = filter_embeddings(emb, seg)
    psi, fea_ref = z[f"vbx/{seed}/psi"], z[f"vbx/{seed}/fea"]
    o_x, o_p, o_psi = vbx_oracle.plda_setup(xt, plda)
    # two inversions and a generalized eigenproblem: their rounding follows the BLAS kernel and thread count (up to
    # 1.5e-10 relative on psi and 3.4e-10 on the features across OpenBLAS's x86 kernels), and the stored reference
    # values were computed with another BLAS build than the one a test run may use
    np.testing.assert_allclose(o_psi, psi, rtol=1e-9)
    np.testing.assert_allclose(o_p(o_x(train), lda_dim=128), fea_ref, rtol=0, atol=2e-9)
    labels = np.random.default_rng(seed).integers(0, 5, size=len(train))
    for Fa, Fb in [(0.07, 0.8), (0.3, 10.0)]:
        g_ref, pi_ref = z[f"vbx/{seed}/{Fa:g}_{Fb:g}/gamma"], z[f"vbx/{seed}/{Fa:g}_{Fb:g}/pi"]
        g, pi, _ = vbx_oracle.vb_gmm(fea_ref, psi[:128], vbx_oracle.init_responsibilities(labels), Fa, Fb, 20)
        np.testing.assert_allclose(g, g_ref, rtol=0, atol=1e-12)
        np.testing.assert_allclose(pi, pi_ref, rtol=0, atol=1e-12)


@pytest.mark.parametrize("seed", range(6))
def test_fcluster_maxclust_equals_scipy(seed):
    from scipy.cluster.hierarchy import fcluster, linkage
    from diarizen_b200.clustering import fcluster_maxclust
    r = np.random.default_rng(seed)
    n = int(r.integers(3, 120))
    x = r.standard_normal((n, 6)) + 3.0 * r.integers(0, 4, size=(n, 1))
    Z = linkage(x, method="centroid", metric="euclidean")
    for t in [1, 2, 3, 5, 9, 30, n - 2, n - 1, n, n + 1, n + 2]:
        if t >= 1:
            np.testing.assert_array_equal(fcluster_maxclust(Z, t), fcluster(Z, t, criterion="maxclust"))


def test_vbx_call_oracle_runs_and_separates():
    xt, plda, emb, seg = _case(3)
    hard, soft, cent = vbx_oracle.vbx_cluster_call(emb, seg, xt, plda, 0.6, 0.07, 0.8)
    assert hard.shape == emb.shape[:2] and soft.shape[:2] == emb.shape[:2]
    assert cent.shape[0] == soft.shape[2] >= 1


def test_host_plda_transform_equals_oracle():
    from diarizen_b200.clustering import PldaTransform
    xt, plda, emb, seg = _case(4)
    from oracle.pipeline_oracle import filter_embeddings
    train, _, _ = filter_embeddings(emb, seg)
    o_x, o_p, o_psi = vbx_oracle.plda_setup(xt, plda)
    tf = PldaTransform(xt, plda)
    np.testing.assert_allclose(tf.psi, o_psi, rtol=1e-13)
    np.testing.assert_allclose(tf(train, 128), o_p(o_x(train), lda_dim=128), rtol=0, atol=1e-11)
    np.testing.assert_allclose(tf(train, 64), o_p(o_x(train), lda_dim=64), rtol=0, atol=1e-11)
