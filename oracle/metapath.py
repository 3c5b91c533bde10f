"""Metapath composition of HAN, restated with numpy / scipy.

HAN/utils/data_utils.py:85-89 (`HeteroGraph.get_mate_path_graph`) builds each metapath adjacency from a relation
matrix P (paper x author, paper x subject) as the binarised product P·Pᵀ, a dense float64 N x N 0/1 array whose
positive entries the attention layers use as the mask.  The reference snapshot ships only `HAN/models`, so this
restatement is the contract the tests hold the device composition (`CSRGraph.pattern_product` / `metapath`) to:
the CSR pattern of (A_bool @ B_bool) > 0, optionally + I, with every row's column ids ascending — the
`nonzero()` order of that dense mask.
"""
import numpy as np
import scipy.sparse as sp


def _pattern(indptr, indices, shape):
    """0/1 scipy CSR of a pattern whose rows may repeat column ids (repeats become one entry)."""
    m = sp.csr_matrix((np.ones(len(indices), dtype=np.int64), np.asarray(indices, dtype=np.int64),
                       np.asarray(indptr, dtype=np.int64)), shape=shape)
    m.sum_duplicates()
    m.data[:] = 1
    return m


def pattern_product(a_indptr, a_indices, b_indptr, b_indices, n_a, k, n_b, row_range=None, self_loops=False):
    """(indptr int64, indices int32) of rows [lo, hi) of pattern(A·B), columns ascending; self_loops adds (i, i)."""
    lo, hi = (0, n_a) if row_range is None else row_range
    A = _pattern(a_indptr, a_indices, (n_a, k))[lo:hi]
    B = _pattern(b_indptr, b_indices, (k, n_b))
    C = (A @ B).tocsr()
    if self_loops:
        assert n_a == n_b, "self_loops needs a square product"
        eye = sp.csr_matrix((np.ones(hi - lo, dtype=np.int64), (np.arange(hi - lo), np.arange(lo, hi))),
                            shape=(hi - lo, n_b))
        C = (C + eye).tocsr()
    C = sp.csr_matrix((C > 0).astype(np.int64))
    C.sort_indices()
    return C.indptr.astype(np.int64), C.indices.astype(np.int32)


def metapath(indptr, indices, n, x, self_loops=False):
    """pattern(R·Rᵀ) (+ I) of a relation R [n x x]: HAN/utils/data_utils.py:85-89 without the dense array."""
    R = _pattern(indptr, indices, (n, x))
    Rt = R.T.tocsr()
    return pattern_product(R.indptr, R.indices, Rt.indptr, Rt.indices, n, x, n, self_loops=self_loops)
