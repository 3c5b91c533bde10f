"""GTN's sparse composition without a GPU: the float64 restatement (oracle/gtn_sparse.py) against the reference's
golden and against the dense restatement (oracle/gtn.py), and the C ABI of the value products refusing bad
arguments before any CUDA call."""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_err
from oracle import gtn as ogtn
from oracle import gtn_sparse as S


def _params(g):
    return {k[6:]: v for k, v in g.items() if k.startswith("param.")}


def test_sparse_oracle_matches_reference_golden():
    g = load_golden("gtn_small.npz")
    y = S.gtn_forward(g["A"], g["X"], g["target"], _params(g), 2, 2)
    assert rel_err(y, g["y"]) < 1e-6


def _random_stack(seed, n, K, density):
    rng = np.random.default_rng(seed)
    A = np.zeros((n, n, K))
    for k in range(K - 1):
        mask = rng.random((n, n)) < density
        A[:, :, k] = mask * rng.uniform(0.1, 1.0, (n, n))
    A[:, :, K - 1] = np.eye(n)  # GTN appends the identity as the last edge type
    A[n - 3:, :, :K - 1] = 0     # rows reached by the identity only
    A[:, n - 2, :K - 1] = 0
    return A


def _dense_H(A, params, C, L):
    """H [C, N, N] of oracle/gtn.py's dense composition in float64 (the loop of gtn_forward)."""
    F = torch.nn.functional
    A = torch.from_numpy(A).unsqueeze(0).permute(0, 3, 1, 2)

    def conv(name):
        return torch.sum(A * F.softmax(torch.from_numpy(params[name]), dim=1), dim=1)

    H = torch.bmm(conv("layers.0.conv1.weight"), conv("layers.0.conv2.weight"))
    for layer in range(1, L):
        H = torch.stack([ogtn.norm(H[c]) for c in range(C)], dim=0)
        H = torch.bmm(H, conv(f"layers.{layer}.conv1.weight"))
    return H.numpy()


@pytest.mark.parametrize("layers", [1, 2, 3])
@pytest.mark.parametrize("seed", [0, 1])
def test_sparse_patterns_and_values_match_dense_composition(layers, seed):
    n, K, C = 40, 4, 3
    A = _random_stack(seed, n, K, 0.04)
    rng = np.random.default_rng(100 + seed)
    params = {f"layers.{l}.conv{j}.weight": rng.standard_normal((C, K, 1, 1)) for l in range(layers) for j in (1, 2)}
    indptr, indices, V = S.union(A)
    (p_ptr, p_idx), H = S.compose((indptr, indices), V, params, layers)
    dense = _dense_H(A, params, C, layers)
    for c in range(C):
        rows, cols = np.nonzero(dense[c])
        assert np.array_equal(p_ptr, np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n))]))
        assert np.array_equal(p_idx, cols)
        assert np.abs(H[:, c] - dense[c][rows, cols]).max() <= 1e-12 * np.abs(dense[c]).max()


def test_drop_diagonal_and_column_normalize():
    ptr, idx, keep = S.drop_diagonal(np.array([0, 2, 3, 5]), np.array([0, 2, 1, 0, 1]))
    assert ptr.tolist() == [0, 1, 1, 3] and idx.tolist() == [2, 0, 1] and keep.tolist() == [1, 3, 4]
    out = S.column_normalize(ptr, idx, np.array([[2.0], [1.0], [4.0]]), 3)
    assert out[:, 0].tolist() == [1.0, 1.0, 1.0]


def test_spgemm_abi_bad_arguments_return_status(lib):
    # checks run before any CUDA call: no device needed
    fake = 256  # a non-null address that is never dereferenced
    fwd = [fake, fake, fake, 4, 4, 8, fake, fake, fake, fake, 4, 8, fake, fake, fake]
    assert lib.gnn_spgemm_values_f32(*fwd, 2, None, None, 0, None) == 5  # no workspace
    assert lib.gnn_spgemm_values_f32(*fwd, 9, None, fake, 1 << 30, None) == 3  # C over the cap
    assert lib.gnn_spgemm_values_f32(*fwd, 0, None, fake, 1 << 30, None) == 1
    bad = list(fwd)
    bad[0] = None
    assert lib.gnn_spgemm_values_f32(*bad, 2, None, fake, 1 << 30, None) == 1
    assert b"null pointer" in lib.gnn_last_error_string()
    bad = list(fwd)
    bad[3] = -1
    assert lib.gnn_spgemm_values_f32(*bad, 2, None, fake, 1 << 30, None) == 1
    bad = list(fwd)
    bad[10] = 1 << 31
    assert lib.gnn_spgemm_values_f32(*bad, 2, None, fake, 1 << 30, None) == 1
    bwd = [fake, fake, fake, 4, 4, 8, fake, fake, fake, fake, fake, fake, 4, 8, fake, fake, fake, fake, fake, fake, 8, 2]
    assert lib.gnn_spgemm_values_bwd_f32(*bwd, fake, fake, None, None, 0, None) == 5
    assert lib.gnn_spgemm_values_bwd_f32(*bwd[:-1], 9, fake, fake, None, fake, 1 << 30, None) == 3
    nul = list(bwd)
    nul[6] = None  # Aᵀ, which dB needs
    assert lib.gnn_spgemm_values_bwd_f32(*nul, None, fake, None, fake, 1 << 30, None) == 1
    nul = list(bwd)
    nul[9] = None  # B's rowptr, which dA needs
    assert lib.gnn_spgemm_values_bwd_f32(*nul, fake, None, None, fake, 1 << 30, None) == 1
    nul = list(bwd)
    nul[19] = None  # dC
    assert lib.gnn_spgemm_values_bwd_f32(*nul, fake, fake, None, fake, 1 << 30, None) == 1
