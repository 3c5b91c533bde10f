"""GTN's learned metapath composition in sparse form, restated with numpy / scipy in float64.

oracle/gtn.py: gtn_forward restates GTN/models/{GTN,GTLayer,GTConv}.py with dense [C, N, N] products.  The same
computation on sparse patterns (DESIGN §4.10), the contract `RelationStack` / `GTN_Model.forward` on a stack are
held to:
  U, V      the union pattern of the K relations (ascending columns) and their values [nnz_U, K], 0 where a relation
            lacks the entry;
  a_c       = V · softmax(w)ᵀ, the values of GTConv's Σ_k s[c, k]·A_k on U;
  P_1 = pattern(U·U),  D_l = P_l without its diagonal,  P_{l+1} = pattern(D_l·U);
  H         values [nnz(P_l), C]; layer 0 a_c(conv1)·b_c(conv2), layer l >= 1 norm(H_c)·a_c(conv1_l), with `norm`
            the column normalisation of the off-diagonal part (GTN.py:7-19, inf -> 0);
  the head  relu(gcn_conv(X, H_c)) per channel, linear1, ReLU, linear2 on target_x.
"""
import numpy as np
import scipy.sparse as sp

from .metapath import pattern_product


def _csr(indptr, indices, data, shape):
    return sp.csr_matrix((data, np.asarray(indices, np.int64), np.asarray(indptr, np.int64)), shape=shape)


def union(A):
    """(indptr, indices, V [nnz_U, K]) of a dense stack A [N, N, K]."""
    A = np.asarray(A, dtype=np.float64)
    rows, cols = np.nonzero((A != 0).any(axis=2))  # row-major: ascending columns within a row
    indptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=A.shape[0]))]).astype(np.int64)
    return indptr, cols.astype(np.int32), A[rows, cols]


def drop_diagonal(indptr, indices):
    """(indptr, indices, kept slots) of a pattern without its diagonal."""
    indptr = np.asarray(indptr, np.int64)
    rows = np.repeat(np.arange(len(indptr) - 1), np.diff(indptr))
    keep = rows != np.asarray(indices)
    cum = np.concatenate([[0], np.cumsum(keep)])
    return cum[indptr].astype(np.int64), np.asarray(indices)[keep].astype(np.int32), np.nonzero(keep)[0]


def patterns(indptr, indices, n, num_layers):
    """[(indptr, indices) of P_l] and [(indptr, indices, kept slots) of D_l], l = 1 .. num_layers."""
    P, D = [], []
    a_ptr, a_idx = indptr, indices
    for _ in range(num_layers):
        p = pattern_product(a_ptr, a_idx, indptr, indices, n, n, n)
        d = drop_diagonal(*p)
        P.append(p)
        D.append(d)
        a_ptr, a_idx = d[0], d[1]
    return P, D


def values_on(M, indptr, indices):
    """The entries of the scipy matrix M at the pattern (indptr, indices), 0 where M has none."""
    M = sp.csr_matrix(M)
    M.sum_duplicates()
    M.sort_indices()
    n_cols = M.shape[1]
    m_keys = np.repeat(np.arange(M.shape[0], dtype=np.int64), np.diff(M.indptr)) * n_cols + M.indices
    rows = np.repeat(np.arange(len(indptr) - 1, dtype=np.int64), np.diff(indptr))
    keys = rows * n_cols + np.asarray(indices, np.int64)
    pos = np.searchsorted(m_keys, keys)
    pos_c = np.minimum(pos, max(len(m_keys) - 1, 0))
    hit = (pos < len(m_keys)) & (m_keys[pos_c] == keys) if len(m_keys) else np.zeros(len(keys), bool)
    out = np.zeros(len(keys))
    out[hit] = M.data[pos_c[hit]]
    return out


def product_values(a_ptr, a_idx, a_val, b_ptr, b_idx, b_val, c_ptr, c_idx, n_a, k, n_b):
    """Values [nnz_C, C] of A·B on the pattern C, channel by channel."""
    a_val, b_val = np.asarray(a_val, np.float64), np.asarray(b_val, np.float64)
    out = np.zeros((len(c_idx), a_val.shape[1]))
    for c in range(a_val.shape[1]):
        M = _csr(a_ptr, a_idx, a_val[:, c], (n_a, k)) @ _csr(b_ptr, b_idx, b_val[:, c], (k, n_b))
        out[:, c] = values_on(M, c_ptr, c_idx)
    return out


def column_normalize(indptr, indices, val, n):
    """val [nnz, C] on a pattern (no diagonal) with every column divided by its sum, inf -> 0 (GTN.py:7-19)."""
    val = np.asarray(val, np.float64)
    sums = np.zeros((n, val.shape[1]))
    np.add.at(sums, np.asarray(indices, np.int64), val)
    with np.errstate(divide="ignore"):
        inv = np.where(sums == 0, 0.0, 1.0 / np.where(sums == 0, 1.0, sums))
    return val * inv[np.asarray(indices, np.int64)]


def softmax_weights(w):
    """softmax(conv.weight[:, :, 0, 0], dim=1) in float64: [C, K]."""
    w = np.asarray(w, np.float64)[:, :, 0, 0]
    e = np.exp(w - w.max(axis=1, keepdims=True))
    return e / e.sum(axis=1, keepdims=True)


def compose(U, V, params, num_layers):
    """(P_L, values H [nnz(P_L), C]) of GTN's composition on the union (U = (indptr, indices))."""
    indptr, indices = U
    n = len(indptr) - 1
    P, D = patterns(indptr, indices, n, num_layers)
    H = None
    for layer in range(num_layers):
        a = V @ softmax_weights(params[f"layers.{layer}.conv1.weight"]).T
        if layer == 0:
            b = V @ softmax_weights(params["layers.0.conv2.weight"]).T
            H = product_values(indptr, indices, a, indptr, indices, b, *P[0], n, n, n)
        else:
            d_ptr, d_idx, keep = D[layer - 1]
            Hn = column_normalize(d_ptr, d_idx, H[keep], n)
            H = product_values(d_ptr, d_idx, Hn, indptr, indices, a, *P[layer], n, n, n)
    return P[-1], H


def gtn_forward(A, X, target_x, params, num_channels, num_layers):
    """GTN_Model.forward (GTN.py:62-88) on the sparse composition, float64: the logits [len(target_x), classes]."""
    params = {k: np.asarray(v, np.float64) for k, v in params.items()}
    X = np.asarray(X, np.float64)
    indptr, indices, V = union(A)
    n = len(indptr) - 1
    (p_ptr, p_idx), H = compose((indptr, indices), V, params, num_layers)
    rows = np.repeat(np.arange(n), np.diff(p_ptr))
    off = rows != p_idx
    XW = X @ params["weight"]
    outs = []
    for c in range(num_channels):
        # gcn_conv (GTN.py:49-52): norm(H, add=True)ᵀ · XW, norm = offdiag + I, columns divided by their sums
        Hp = sp.csr_matrix((H[off, c], (rows[off], p_idx[off])), shape=(n, n)) + sp.identity(n)
        deg = np.asarray(Hp.sum(axis=0)).ravel()
        inv = np.where(deg == 0, 0.0, 1.0 / np.where(deg == 0, 1.0, deg))
        outs.append(np.maximum((Hp @ sp.diags(inv)).T @ XW, 0.0))
    X_ = np.maximum(np.concatenate(outs, axis=1) @ params["linear1.weight"].T + params["linear1.bias"], 0.0)
    return X_[np.asarray(target_x)] @ params["linear2.weight"].T + params["linear2.bias"]
