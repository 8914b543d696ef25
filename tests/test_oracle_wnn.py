"""CPU: groundwork for the WNN row (SURVEY 8f-f1, round 2).  The reference's own ``neighbors`` driver
(muon/_core/preproc.py:264-640) runs in the build container with exact stand-ins for its third-party imports
(oracle/_third_party.py); these tests pin the stand-ins and the committed golden."""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import golden_csr, load_golden
from oracle import _third_party as tp


def test_exact_search_and_helpers():
    rng = np.random.default_rng(0)
    X = rng.normal(size=(60, 5))
    idx, dist, _ = tp.nearest_neighbors(X, 7, "euclidean")
    D = np.linalg.norm(X[:, None] - X[None], axis=-1)
    np.testing.assert_array_equal(idx[:, 0], np.arange(60))             # self first, distance 0
    np.testing.assert_allclose(dist, np.sort(D, axis=1)[:, :7], rtol=1e-12)
    a, b = np.array([1, 4, 7, 9]), np.array([2, 4, 9, 11, 12])
    assert tp.sparse_jaccard(a, None, b, None) == pytest.approx(1 - 2 / 7)
    assert tp.sparse_euclidean(a, np.ones(4), b, np.ones(5)) == pytest.approx(np.sqrt(5))
    assert tp.euclidean(X[0], X[1]) == pytest.approx(D[0, 1])


def test_umap_connectivities_properties():
    rng = np.random.default_rng(1)
    X = rng.normal(size=(80, 4))
    idx, dist, _ = tp.nearest_neighbors(X, 10, "euclidean")
    C = tp.umap_connectivities(idx, dist, n_obs=80, n_neighbors=10)
    assert sp.isspmatrix_csr(C) and (C != C.T).nnz == 0                  # fuzzy union is symmetric
    assert C.data.min() > 0 and C.data.max() <= 1.0 + 1e-6
    assert C.diagonal().sum() == 0
    # each point's nearest non-self neighbour has membership 1 (local_connectivity = 1)
    nearest = idx[:, 1]
    assert np.allclose(np.asarray(C[np.arange(80), nearest]).ravel(), 1.0, atol=1e-6)


def test_wnn_golden_is_consistent():
    z = load_golden("wnn_small.npz")
    n = z["rep_rna"].shape[0]
    w = z["w_rna"] + z["w_atac"]
    np.testing.assert_allclose(w, 1.0, rtol=1e-12)                       # softmax over modalities
    Dm = golden_csr(z, "wnn_dist")
    k = int(z["n_neighbors"])
    assert Dm.shape == (n, n) and np.all(np.diff(Dm.indptr) == k + 1)    # preproc.py:604: top (n_neighbors+1) per row
    assert Dm.data.min() >= 0 and Dm.data.max() <= np.sqrt(0.5) + 1e-12  # sqrt(0.5 (1 - affinity)), affinity in [0,1]
    Cm = golden_csr(z, "wnn_conn")
    assert (Cm != Cm.T).nnz == 0


def test_numpy_restatement_reproduces_reference_driver_golden():
    from oracle.wnn_ref import wnn_ref
    z = load_golden("wnn_small.npz")
    r = wnn_ref([z["rep_rna"], z["rep_atac"]], [golden_csr(z, "knn_rna"), golden_csr(z, "knn_atac")],
                int(z["n_neighbors"]), n_multineighbors=40)
    np.testing.assert_allclose(r["weights"][:, 0], z["w_rna"], rtol=1e-12)
    got = r["distances"].copy()
    got.sort_indices()
    ref = golden_csr(z, "wnn_dist")
    np.testing.assert_array_equal(got.indices, ref.indices)
    np.testing.assert_allclose(got.data, ref.data, rtol=1e-10, atol=1e-14)
    assert abs(r["connectivities"] - golden_csr(z, "wnn_conn")).max() < 1e-6


def test_product_umap_connectivities_match_the_standin_on_cpu_tensors():
    """muon_b200.pp._umap_connectivities is plain torch (no custom kernel), so its arithmetic can be checked without
    a GPU against oracle/_third_party.py::umap_connectivities (= scanpy's umap connectivities wrapper)."""
    import torch
    from muon_b200.pp import _umap_connectivities
    from oracle import _third_party as tp
    rng = np.random.default_rng(5)
    n, k = 300, 12
    X = rng.normal(size=(n, 6)) + 3.0 * np.eye(6)[rng.integers(0, 6, n)]
    idx, dist, _ = tp.nearest_neighbors(X, k, "euclidean")
    dist = dist.astype(np.float32)
    dist[7, 1:4] = dist[7, 1]                       # ties at rho
    idx[11, -1] = -1                                # a missing neighbour slot
    ref = tp.umap_connectivities(idx, dist, n_obs=n, n_neighbors=k)
    got = _umap_connectivities(torch.from_numpy(idx), torch.from_numpy(dist), n)
    assert (got != got.T).nnz == 0
    assert abs(got - ref).max() < 2e-5
    assert got.nnz == ref.nnz
