"""Golden fixture for the LSI parity test at BASELINE configs[1]'s width (200k peaks).

Runs the CPU oracle -- ``oracle.tfidf_ref`` (restated preproc.py:92-119) then float64
``scipy.sparse.linalg.svds`` with muon's post-processing (``oracle.lsi_ref``, tools.py:53-65) -- on the
first N_CELLS rows of the benchmark's synthetic matrix (same generator, tables and seed as bench.py), in
the build container (takes a few minutes of single-threaded ARPACK, which is why the result is a fixture):

    python tests/golden/make_golden_lsi_slice.py

Outputs (committed): ``lsi_slice_20k.npz`` holds the singular values (k+1, float64), V on 4096 evenly spaced
peaks and checksums of the input so the GPU test can prove it regenerated the same matrix;
``lsi_slice_20k_U.npz`` holds U on 4096 evenly spaced cells.  Factors are stored as float32 of the float64
result, and sampled so that each file stays under 1 MB.
"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from muon_b200._synth import generate_host, make_tables  # noqa: E402
from oracle.lsi_ref import lsi_ref  # noqa: E402
from oracle.tfidf_ref import tfidf_ref  # noqa: E402

N_CELLS, N_PEAKS, DENSITY, TOPICS, SEED, K = 20_000, 200_000, 0.03, 64, 1, 50
OUT = os.path.dirname(os.path.abspath(__file__))


def main():
    tb = make_tables(N_PEAKS, DENSITY, TOPICS, SEED)
    t0 = time.time()
    C = generate_host(N_CELLS, N_PEAKS, DENSITY, tables=tb, row0=0)
    print("generated", C.shape, C.nnz, f"{time.time() - t0:.1f}s", flush=True)
    X = tfidf_ref(C)
    X.sort_indices()
    t0 = time.time()
    r = lsi_ref(X, K + 1, scale_embeddings=False, dtype=np.float64)
    print("svds", f"{time.time() - t0:.1f}s", r["svalues"][:5], flush=True)
    rows = np.unique(np.linspace(0, N_PEAKS - 1, 4096).astype(np.int64))
    np.savez_compressed(
        os.path.join(OUT, "lsi_slice_20k.npz"),
        shape=np.array([N_CELLS, N_PEAKS]), density=DENSITY, topics=TOPICS, seed=SEED, k=K,
        svalues=r["svalues"], V_rows=rows,
        V_sample=r["LSI"][rows, :K].astype(np.float32),
        nnz=C.nnz, counts_sum=float(C.data.astype(np.float64).sum()),
        tfidf_sum=float(X.data.astype(np.float64).sum()), indices_sum=int(C.indices.astype(np.int64).sum()))
    cells = np.unique(np.linspace(0, N_CELLS - 1, 4096).astype(np.int64))
    np.savez_compressed(os.path.join(OUT, "lsi_slice_20k_U.npz"), U_rows=cells,
                        U_sample=r["U"][cells, :K].astype(np.float32))


if __name__ == "__main__":
    main()
