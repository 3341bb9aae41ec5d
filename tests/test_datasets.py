"""datasets.py (MAT-file loading + the scripts' preprocessing) against the committed fixtures.  The reference's data
files are read from a checkout of the reference named by KR_REFERENCE_DIR; the preprocessing helpers are also tested
stand-alone."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import load_graph

REF = os.environ.get("KR_REFERENCE_DIR", "")
needs_ref = pytest.mark.skipif(not (REF and os.path.isdir(REF)), reason="KR_REFERENCE_DIR names no checkout of the reference")


def test_unweighted_preprocessing_on_a_toy_graph():
    from krylov_robustness_b200.datasets import unweighted_adjacency
    # directed, weighted, with a self loop and two components (sizes 3 and 2): keep the triangle
    A = sp.csr_matrix((np.array([2.0, 5.0, 1.0, 7.0, 3.0]), (np.array([0, 1, 2, 3, 1]), np.array([1, 2, 0, 4, 1]))), shape=(5, 5))
    B = unweighted_adjacency(A)
    assert B.shape == (3, 3) and B.nnz == 6 and (B != B.T).nnz == 0
    assert B.diagonal().sum() == 0 and set(B.data) == {1.0}


@needs_ref
def test_loaders_reproduce_the_fixtures():
    from krylov_robustness_b200 import datasets as D
    for name, path in (("transport_Anaheim", "datasets_paper/Transport/Anaheim.mat"),
                       ("transport_Rome", "datasets_paper/Transport/Rome.mat")):
        A = D.load_problem(os.path.join(REF, path))
        F = load_graph(name)
        assert A.shape == F.shape and (A != F).nnz == 0
    A0 = D.load_problem(os.path.join(REF, "MIOBI Codes", "dt_oregon.mat") + "::A0", unweighted=False)
    assert (A0 != load_graph("oregon_A0")).nnz == 0
    grids = D.load_power_grids(os.path.join(REF, "datasets_paper", "voltage_adjacencies_average_2.mat"), ["Sweden", "England"])
    for k, A in grids.items():
        F = load_graph("grid_" + k)
        assert A.shape == F.shape and abs(A - F).max() <= 1e-15


@needs_ref
def test_v73_files_through_the_minimal_hdf5_reader():
    """CollegeMsg, Drugs, as_735 are MATLAB v7.3 (HDF5) files; the image has no HDF5 library, hdf5_min.py reads them.
    Two of them carry the symmetrised pattern a second time (variable W, written by a different code path of MATLAB):
    what comes out of Problem.A after the scripts' preprocessing must be exactly that."""
    from krylov_robustness_b200 import datasets as D
    from krylov_robustness_b200.hdf5_min import loadmat73, is_v73
    shapes = {"Drugs": 616, "CollegeMsg": 1899, "as_735": 7716}
    for name, n in shapes.items():
        path = os.path.join(REF, "datasets_paper", "Misc", name + ".mat")
        assert is_v73(path)
        raw = loadmat73(path)
        P = raw["Problem"]
        assert sp.issparse(P["A"]) and P["A"].shape == (n, n) and isinstance(P["name"], str) and len(P["name"]) > 3
        A = D.load_problem(path)
        assert (A != A.T).nnz == 0 and set(A.data) == {1.0} and A.diagonal().sum() == 0
        F = load_graph("misc_" + name)
        assert A.shape == F.shape and (A != F).nnz == 0
        if "W" in raw:
            S = sp.csr_matrix(P["A"])
            S = (S + S.T).tocsr()
            S.data[:] = 1.0
            S.setdiag(0)
            S.eliminate_zeros()
            assert (S != sp.csr_matrix(raw["W"])).nnz == 0
    assert not is_v73(os.path.join(REF, "datasets_paper", "Misc", "jazz.mat"))


def test_hdf5_reader_rejects_what_it_does_not_understand(tmp_path):
    """No reference files needed: a MAT-v5 header is not v7.3, and a file without an HDF5 signature or with a newer
    superblock version raises Hdf5Error instead of returning garbage."""
    from krylov_robustness_b200.hdf5_min import Hdf5Error, is_v73, loadmat73
    import scipy.io as sio
    v5 = tmp_path / "v5.mat"
    sio.savemat(str(v5), {"A": sp.identity(3, format="csc")})
    assert not is_v73(str(v5))
    bad = tmp_path / "bad.mat"
    bad.write_bytes(b"MATLAB 7.3 MAT-file, Platform: none".ljust(512, b" ") + b"not hdf5 at all" * 10)
    assert is_v73(str(bad))
    with pytest.raises(Hdf5Error, match="signature"):
        loadmat73(str(bad))
    newer = tmp_path / "newer.mat"
    newer.write_bytes(b"MATLAB 7.3 MAT-file".ljust(512, b" ") + b"\x89HDF\r\n\x1a\n" + bytes([2]) + b"\0" * 64)
    with pytest.raises(Hdf5Error, match="superblock version 2"):
        loadmat73(str(newer))
