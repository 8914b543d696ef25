"""GPU tests added in round 2: staging engine + fingerprints, half-operand SpMM, the LSI driver's cheaper
schedules (no final Rayleigh-Ritz pass, half-precision first phase), LSI at configs[1]'s width against a
float64 svds fixture (panelled A^T, 64-bit non-zero offsets), the pipelined host path of tfidf()."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import muon_b200 as mu
from conftest import load_golden
from muon_b200 import _device
from muon_b200._containers import SimpleAnnData
from muon_b200._synth import generate_device, generate_host, make_tables
from oracle.lsi_ref import compare_lsi, lsi_ref, sign_align
from oracle.tfidf_ref import tfidf_ref

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------
def test_stager_roundtrip_narrowing_and_fingerprints(cuda):
    rng = np.random.default_rng(0)
    st = _device.Stager(threads=5)
    n = (_device._STAGE_BYTES // 4) * 5 + 12345          # > n_bufs chunks: ring reuse is exercised
    a = rng.integers(0, 2**31 - 1, n, dtype=np.int64)
    d = torch.empty(n, dtype=torch.int32, device=cuda)
    h = st.h2d(a, d, narrow=True, want_hash=True)
    torch.cuda.synchronize()
    assert np.array_equal(d.cpu().numpy(), a.astype(np.int32))
    assert h == st.fingerprint(a) == st.fingerprint(a.astype(np.int32)) == _device.device_fingerprint(d)
    cuts = [(0, 1000), (1000, n // 2), (n // 2, n)]
    assert _device.device_fingerprints(d, cuts) == [st.fingerprint(a[k0:k1]) for k0, k1 in cuts]
    back = np.empty(n, dtype=np.int32)
    h2 = st.d2h(d, back, want_hash=True)
    assert h2 == h and np.array_equal(back, a.astype(np.int32))
    # float payload, no hash; then an immediately following transfer on another stream (buffer guards)
    f = rng.standard_normal(n).astype(np.float32)
    df = torch.empty(n, dtype=torch.float32, device=cuda)
    side = torch.cuda.Stream()
    st.h2d(f, df, stream=side)
    st.h2d(a[:1000], d[:1000], narrow=True)
    torch.cuda.synchronize()
    assert np.array_equal(df.cpu().numpy(), f)
    # position dependence: swapping two elements or editing one changes the fingerprint
    b = a.copy()
    b[[3, 77777]] = b[[77777, 3]]
    assert st.fingerprint(b) != h
    c = a.copy()
    c[n - 1] ^= 1
    assert st.fingerprint(c) != h
    with pytest.raises(_device.MuonB200Error):
        st.h2d(np.array([2**40] * 10, dtype=np.int64), d[:10], narrow=True)


def test_to_device_to_host_large(cuda):
    rng = np.random.default_rng(1)
    x = rng.standard_normal(5_000_000).astype(np.float64)          # 40 MB: staged path, 8-byte elements
    t = _device.to_device(x, cuda)
    assert t.dtype == torch.float64 and np.array_equal(_device.to_host(t), x)
    i = rng.integers(0, 1000, 6_000_000, dtype=np.int64)
    ti = _device.to_device(i, cuda, np.int32)
    assert ti.dtype == torch.int32 and np.array_equal(ti.cpu().numpy(), i.astype(np.int32))
    u = rng.integers(0, 60000, 9_000_000).astype(np.uint16)       # odd dtype: raw upload + device conversion
    tu = _device.to_device(u, cuda, np.float32)
    assert tu.dtype == torch.float32 and np.array_equal(tu.cpu().numpy(), u.astype(np.float32))


# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("P", [32, 64, 128])
def test_spmm_half_operand(cuda, P):
    """C = A @ half(B) with fp32 accumulation: equal to the float64 product with the SAME rounded operand to
    fp32 summation accuracy, for the CSR layout and the pair layout (transposed panels)."""
    X = tfidf_ref(generate_host(700, 900, 0.06, n_topics=6, seed=5)).astype(np.float32)
    X.sort_indices()
    A = mu.DeviceCSR.from_scipy(X)
    g = torch.Generator(device=cuda).manual_seed(0)
    B = torch.randn((900, P), generator=g, device=cuda) / 30.0
    Bh = _device.to_half_scaled(B)
    Bh_ref = Bh.cpu().numpy().astype(np.float64) / _device.HALF_SCALE
    assert np.abs(Bh_ref - B.cpu().numpy()).max() < 2.0 ** -11 * np.abs(B.cpu().numpy()).max() * 1.01
    ref = X.astype(np.float64) @ Bh_ref
    for dyn in (False, True):
        C = _device.spmm_h16(A, Bh, dynamic=dyn).cpu().numpy()
        assert np.abs(C - ref).max() <= 2e-6 * np.abs(ref).max()
    C2 = _device.spmm_h16(A, Bh, out=torch.ones((700, P), device=cuda), accumulate=True).cpu().numpy()
    assert np.abs(C2 - 1.0 - ref).max() <= 3e-6 * max(1.0, np.abs(ref).max())
    # pair layout: (A^T) @ half(U)
    U = torch.randn((700, P), generator=g, device=cuda) / 25.0
    Tp = _device.TransposedPanels(A, P)
    W = Tp.spmm(U, half=True).cpu().numpy()
    Uh = _device.to_half_scaled(U).cpu().numpy().astype(np.float64) / _device.HALF_SCALE
    refT = X.T.astype(np.float64) @ Uh
    assert np.abs(W - refT).max() <= 2e-6 * np.abs(refT).max()


@pytest.mark.parametrize("polish,lowp_tol", [(True, 0.0), (False, 0.0), (True, 1e-3), (False, 1e-3)])
@pytest.mark.parametrize("shape,k", [((3000, 2000), 15), ((2500, 1500), 60)])
def test_lsi_cheaper_schedules_vs_svds_float64_truth(cuda, monkeypatch, shape, k, polish, lowp_tol):
    """The driver's cheaper schedules meet the same parity bar as the default: no final Rayleigh-Ritz pass
    (U from the stored left Lanczos blocks), half-precision first phase, and both."""
    monkeypatch.setenv("MUON_B200_LSI_POLISH", "1" if polish else "0")
    monkeypatch.setenv("MUON_B200_LSI_LOWP_TOL", str(lowp_tol))
    n, d = shape
    X = tfidf_ref(generate_host(n, d, 0.05, n_topics=24, seed=n)).astype(np.float32)
    X.sort_indices()
    ref = lsi_ref(X, k + 1, scale_embeddings=False, dtype=np.float64)
    s_next = ref["svalues"][k]
    ref = {"svalues": ref["svalues"][:k], "U": ref["U"][:, :k], "LSI": ref["LSI"][:, :k]}
    a = SimpleAnnData(X.copy())
    info = mu.atac.tl.lsi(a, n_comps=k, scale_embeddings=False, return_info=True)
    assert info.converged
    assert (info.lowp_passes > 0) == (lowp_tol > 0)
    got = {"svalues": a.uns["lsi"]["stdev"].astype(np.float64) * np.sqrt(n - 1), "U": a.obsm["X_lsi"],
           "LSI": a.varm["LSI"]}
    out = compare_lsi(got, ref, rtol=1e-4, s_next=s_next)
    assert out["sigma_rel"] < 1e-5
    Uo = a.obsm["X_lsi"].astype(np.float64)
    assert np.abs(Uo.T @ Uo - np.eye(k)).max() < 1e-5


# ---------------------------------------------------------------------------------------------------------
def _slice_case(cuda):
    z = load_golden("lsi_slice_20k.npz")
    n, d = (int(v) for v in z["shape"])
    tb = make_tables(d, float(z["density"]), int(z["topics"]), int(z["seed"]))
    C = generate_device(n, d, float(z["density"]), tables=tb, row0=0, n_total=n)
    assert C.nnz == int(z["nnz"])                                   # same matrix as the fixture's generator run
    assert float(C.data.sum(dtype=torch.float64)) == float(z["counts_sum"])
    assert int(C.indices.sum(dtype=torch.int64)) == int(z["indices_sum"])
    return z, n, d, C


def _check_slice(z, n, ad, rtol=1e-4):
    k = int(z["k"])
    s_ref = z["svalues"]
    got_s = ad.uns["lsi"]["stdev"].astype(np.float64) * np.sqrt(n - 1)
    zu = load_golden("lsi_slice_20k_U.npz")
    Uref = zu["U_sample"].astype(np.float64)
    Ugot = ad.obsm["X_lsi"][zu["U_rows"]]
    V = ad.varm["LSI"]
    rows = z["V_rows"]
    # singular values: all of them; U: the full gap-aware comparison on the fixture's 4096 sampled cells; V: on its
    # 4096 sampled peaks, sign-aligned through U (v_i and u_i flip together)
    got = {"svalues": got_s, "U": Ugot, "LSI": Ugot}
    ref = {"svalues": s_ref[:k], "U": Uref, "LSI": Uref}
    out = compare_lsi(got, ref, rtol=rtol, s_next=s_ref[k])
    sgn = np.sign(np.sum(Ugot.astype(np.float64) * Uref, axis=0))
    Vs = V[rows].astype(np.float64) * sgn
    Vr = z["V_sample"].astype(np.float64)
    ext = np.concatenate([s_ref[:k], [s_ref[k]]])
    gaps = np.minimum(np.abs(np.diff(ext)), np.concatenate([[np.inf], np.abs(np.diff(ext))[:-1]])) / ext[:-1]
    res = gaps > 5e-3
    e = np.linalg.norm(Vs - Vr, axis=0) / np.linalg.norm(Vr, axis=0)
    assert e[res].max() <= 10 * rtol, f"V rows: {e[res].max():.2e}"      # 4096-row sample of unit vectors in R^200000
    out["V_sample_err"] = float(e[res].max())
    return out


def test_lsi_configs1_width_slice_vs_float64_svds_fixture(cuda, monkeypatch):
    """20 000 cells x 200 000 peaks (1.2e8 nnz) of the benchmark matrix: TF-IDF + LSI k=50 against the committed
    float64 svds result (tests/golden/make_golden_lsi_slice.py), with A^T cut into several row panels."""
    z, n, d, C = _slice_case(cuda)
    monkeypatch.setattr(_device.TransposedPanels, "L2_BUDGET", 1 << 20)       # 4096 cells per panel -> 5 panels
    ad = SimpleAnnData(C)
    mu.atac.pp.tfidf(ad)
    assert abs(float(ad.X.data.sum(dtype=torch.float64)) - float(z["tfidf_sum"])) <= 1e-6 * float(z["tfidf_sum"])
    info = mu.atac.tl.lsi(ad, n_comps=int(z["k"]), scale_embeddings=False, return_info=True)
    assert info.converged and len(ad.X._tp[1].panels) >= 4
    out = _check_slice(z, n, ad)
    assert out["sigma_rel"] < 1e-5
    print("slice parity:", out, "passes", info.passes)


def test_lsi_slice_with_nonzero_offsets_beyond_2_31(cuda):
    """The same slice stored at the END of index/value arrays longer than 2^31 entries, so every non-zero offset
    the kernels compute (indptr values, panel offsets) exceeds int32 -- checked against the same svds fixture."""
    z, n, d, C = _slice_case(cuda)
    base = (1 << 31) + 12_345_678
    nnz = C.nnz
    big_idx = torch.empty(base + nnz, dtype=torch.int32, device=cuda)
    big_val = torch.empty(base + nnz, dtype=torch.float32, device=cuda)
    big_idx[:base].fill_(-1)                                          # poison: reading below the base would fault / corrupt
    big_val[:base].fill_(float("nan"))
    big_idx[base:] = C.indices
    big_val[base:] = C.data
    A = mu.DeviceCSR(C.indptr + base, big_idx, big_val, (n, d))
    A_nnz_view = A.with_data(big_val)                                  # nnz property counts the padded arrays; kernels only use indptr
    del C
    ad = SimpleAnnData(A_nnz_view)
    mu.atac.pp.tfidf(ad)
    mu.atac.tl.lsi(ad, n_comps=int(z["k"]), scale_embeddings=False)
    out = _check_slice(z, n, ad)
    assert out["sigma_rel"] < 1e-5


# ---------------------------------------------------------------------------------------------------------
def test_host_path_pipeline_blocks_and_twin_validation(cuda, monkeypatch):
    """tfidf() on a host matrix: several upload/download blocks, int64 and int32 host indices, result equal to the
    one-shot device path bit for bit; the device twin is reused by lsi() only while EVERY host element is intact."""
    monkeypatch.setattr(_device, "_BLOCK_NNZ", 50_000)
    C = generate_host(3000, 900, 0.05, n_topics=8, seed=4)
    ref = _device.tfidf_csr(mu.DeviceCSR.from_scipy(C)).get()
    for idt in (np.int32, np.int64):
        X = sp.csr_matrix(C.shape, dtype=np.float32)
        X.data, X.indices, X.indptr = C.data.copy(), C.indices.astype(idt), C.indptr.astype(idt)
        ad = SimpleAnnData(X)
        mu.atac.pp.tfidf(ad)
        assert ad.X.indices.dtype == idt and ad.X.indices is X.indices      # replaces its source: arrays shared
        np.testing.assert_array_equal(ad.X.data, ref.data)
        assert len(getattr(ad.X, _device._RESIDENT_ATTR)[1]["blocks"]) >= 3
        assert _device.recall_resident(ad.X) is not None
        # (a) one value edited, (b) two values swapped, (c) one column index edited, (d) indptr edited
        v = ad.X.data[1234]
        ad.X.data[1234] = v * 1.5
        assert _device.recall_resident(ad.X) is None
        ad.X.data[1234] = v
        assert _device.recall_resident(ad.X) is not None
        ad.X.data[[10, 20]] = ad.X.data[[20, 10]]
        assert _device.recall_resident(ad.X) is None
        ad.X.data[[10, 20]] = ad.X.data[[20, 10]]
        j = ad.X.indices[5000]
        ad.X.indices[5000] = j + 1 if j + 1 < 900 else j - 1
        assert _device.recall_resident(ad.X) is None
        ad.X.indices[5000] = j
        assert _device.recall_resident(ad.X) is not None
    # values that are not small integers take the float32 route over the bus (first block decides), same result
    H = C.copy()
    H.data = (H.data * np.float32(0.5)).astype(np.float32)
    np.testing.assert_array_equal(mu.atac.pp.tfidf(SimpleAnnData(H.copy()), inplace=False).data,
                                  _device.tfidf_csr(mu.DeviceCSR.from_scipy(H)).get().data)
    Hm = C.copy()
    Hm.data[-5] = 300.0                                  # only the LAST block falls back
    np.testing.assert_array_equal(mu.atac.pp.tfidf(SimpleAnnData(Hm.copy()), inplace=False).data,
                                  _device.tfidf_csr(mu.DeviceCSR.from_scipy(Hm)).get().data)
    # the result keeps its own index arrays when the source stays alive
    out = mu.atac.pp.tfidf(SimpleAnnData(C), inplace=False)
    assert out.indices is not C.indices and out.indptr is not C.indptr
    np.testing.assert_array_equal(out.data, ref.data)
    # twins can be switched off and released (also all at once: the registry must see unhashable scipy matrices)
    assert _device.release_resident(ad) and _device.recall_resident(ad.X) is None
    ad3 = SimpleAnnData(C.copy())
    mu.atac.pp.tfidf(ad3)
    assert _device.recall_resident(ad3.X) is not None and _device.release_all_resident() >= 1
    assert _device.recall_resident(ad3.X) is None
    # host result buffers are recycled once nothing references them, never while a view is alive
    big = _device._ARENA.empty(40_000_000, np.float32)
    keep = big[5:10]
    addr = big.ctypes.data
    del big
    assert _device._ARENA.empty(40_000_000, np.float32).ctypes.data != addr       # `keep` still pins the block
    del keep
    assert _device._ARENA.empty(40_000_000, np.float32).ctypes.data == addr
    monkeypatch.setenv("MUON_B200_RESIDENT", "0")
    ad2 = SimpleAnnData(C.copy())
    mu.atac.pp.tfidf(ad2)
    assert getattr(ad2.X, _device._RESIDENT_ATTR, None) is None


# ---------------------------------------------------------------------------------------------------------
def test_tiled_reduce_equals_atomic_reduce_and_counts_feed_the_transposition(cuda, monkeypatch):
    """The shared-memory tiled reduce pass: row sums / column sums bit-identical to the one-atomic-per-non-zero
    kernel (integer-valued counts: every order gives the same fp32 sum), entry counts per (row chunk, column)
    equal to a bincount, panels built from those counts identical to panels built by the counting pass, and the
    canonical-form verdict (unsorted row, explicit zero) unchanged."""
    from muon_b200._lib import call, ptr, stream_ptr
    C = generate_host(5000, 30000, 0.03, n_topics=8, seed=9)         # 3 column tiles, 10 row blocks
    A = mu.DeviceCSR.from_scipy(C)
    n, d = C.shape
    monkeypatch.setenv("MUON_B200_TFIDF_TILED", "0")
    ref = _device.tfidf_csr(A)
    monkeypatch.setenv("MUON_B200_TFIDF_TILED", "1")
    got = _device.tfidf_csr(A)
    for key in ("row_sum", "col_sum", "idf"):
        assert torch.equal(ref._aux[key], got._aux[key]), key
    assert torch.equal(ref.data, got.data) and "col_counts" not in ref._aux
    bounds, counts = got._aux["col_counts"]
    assert bounds[0] == 0 and bounds[-1] == n and all(b % _device.tile_rows() == 0 or b == n for b in bounds)
    for c in range(_device.N_CHUNKS):
        lo, hi = int(C.indptr[bounds[c]]), int(C.indptr[bounds[c + 1]])
        want = np.bincount(C.indices[lo:hi], minlength=d)
        assert np.array_equal(counts[c].cpu().numpy(), want), c
    # transposed panels from the reused counts == panels from the counting pass (same indptr; same entry SETS per row)
    monkeypatch.setattr(_device.TransposedPanels, "L2_BUDGET", 1 << 18)       # 1024 cells per panel at pad 64 -> 8 panels
    monkeypatch.setenv("MUON_B200_FILL_TILED", "1")             # the atomic-free fill (opt-in: measured slower at scale)
    Tp = _device.TransposedPanels(got, 64)
    Tq = _device.TransposedPanels(ref, 64)
    assert Tp.counts_reused and Tp.tiled_fill and not Tq.counts_reused and not Tq.tiled_fill
    assert len(Tp.panels) == len(Tq.panels) >= 4
    monkeypatch.setenv("MUON_B200_FILL_TILED", "0")
    Tr = _device.TransposedPanels(got, 64)                       # reused counts, atomic-cursor fill
    assert Tr.counts_reused and not Tr.tiled_fill
    for (a0, a1, Ta), (b0, b1, Tb) in zip(Tp.panels, Tr.panels):
        # same ENTRIES per transposed row ((peak, cell) is unique): order by (peak, cell) and compare cells and value bits
        assert torch.equal(Ta.indptr, Tb.indptr)
        rows = torch.repeat_interleave(torch.arange(d, device=cuda), Ta.indptr[1:] - Ta.indptr[:-1])
        ka = rows * (1 << 20) + Ta.pairs[:, 0].to(torch.int64)
        kb = rows * (1 << 20) + Tb.pairs[:, 0].to(torch.int64)
        oa, ob = torch.argsort(ka), torch.argsort(kb)
        assert torch.equal(ka[oa], kb[ob]) and torch.equal(Ta.pairs[oa, 1], Tb.pairs[ob, 1])
        assert int(Ta.pairs[:, 0].min()) >= 0 and int(Ta.pairs[:, 0].max()) < a1 - a0
    for (a0, a1, Ta), (b0, b1, Tb) in zip(Tp.panels, Tq.panels):
        assert (a0, a1) == (b0, b1) and torch.equal(Ta.indptr, Tb.indptr)
        Y = torch.randn((a1 - a0, 64), device=cuda)
        ya, yb = _device.spmm(Ta, Y).cpu().numpy(), _device.spmm(Tb, Y).cpu().numpy()
        assert np.abs(ya - yb).max() <= 1e-5 * np.abs(yb).max()       # same entry sets, different summation order
    # binarize fused, float sums exact
    gb = _device.tfidf_csr(A, binarize=True)
    monkeypatch.setenv("MUON_B200_TFIDF_TILED", "0")
    rb = _device.tfidf_csr(A, binarize=True)
    assert torch.equal(gb.data, rb.data)
    monkeypatch.setenv("MUON_B200_TFIDF_TILED", "1")
    # an unsorted row: flagged (check_canonical) / silently handled by the order-agnostic kernel (device input)
    Xu = C.copy()
    a = Xu.indptr[777]
    Xu.indices[a:a + 2] = C.indices[a:a + 2][::-1].copy()
    Xu.data[a:a + 2] = C.data[a:a + 2][::-1].copy()
    Au = mu.DeviceCSR.from_scipy(Xu)
    assert _device.tfidf_csr(Au, check_canonical=True) is None
    Au2 = mu.DeviceCSR.from_scipy(Xu)
    out = _device.tfidf_csr(Au2)
    assert not Au2.sorted_indices and torch.equal(out._aux["col_sum"], ref._aux["col_sum"])
    # explicit zero: flagged under check_canonical, harmless otherwise
    Xz = C.copy()
    Xz.data[12345] = 0.0
    assert _device.tfidf_csr(mu.DeviceCSR.from_scipy(Xz), check_canonical=True) is None
    # index beyond n_cols is reported as non-canonical instead of corrupting shared memory
    Xo = C.copy()
    Xo.indices[Xo.indptr[100 + 1] - 1] = d + 5
    st = torch.zeros(1, dtype=torch.int32, device=cuda)
    Ao = mu.DeviceCSR.from_scipy(Xo)
    rs, cs = torch.empty(n, device=cuda), torch.zeros(d, device=cuda)
    call("mub_tfidf_reduce_tiled_f32", ptr(Ao.indptr), ptr(Ao.indices), ptr(Ao.data), n, d, ptr(rs), ptr(cs), ptr(st), 0,
         None, None, 0, 0, None, stream_ptr())
    assert int(st[0]) & 1
