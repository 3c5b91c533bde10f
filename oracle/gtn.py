"""CPU restatement of the GTN pieces next to the hot path (test infrastructure: imported by tests/ only).

  norm      GTN/models/GTN.py:7-19   column normalisation of the learned adjacency
  gcn_conv  GTN/models/GTN.py:49-52  GCN over the learned adjacency
Pinned against the unmodified reference by tests/golden/gtn_small.npz (made by tests/golden/make_golden.py)
and by tests/test_oracle_vs_reference_live.py on fresh seeds."""
import torch


def norm(H: torch.Tensor, add: bool = False) -> torch.Tensor:
    """GTN.py:7-19: H' = offdiag(H) (+ I when add); every column j of H' divided by its sum (inf -> 0)."""
    n = H.shape[0]
    Hp = H * (1.0 - torch.eye(n, dtype=H.dtype))
    if add:
        Hp = Hp + torch.eye(n, dtype=H.dtype)
    deg = Hp.sum(dim=0)                       # column sums == row sums of H'.t() (GTN.py:13)
    inv = deg.pow(-1)
    inv = torch.where(torch.isinf(inv), torch.zeros_like(inv), inv)
    return Hp * inv.unsqueeze(0)


def gcn_conv(X: torch.Tensor, H: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
    """GTN.py:49-52: norm(H, add=True).t() @ (X @ weight)."""
    return norm(H, add=True).t() @ (X @ weight)


def gtn_forward(A, X, target_x, params, num_channels, num_layers):
    """GTN_Model.forward (GTN.py:62-88) with the state_dict `params` (GTConv.py:22, GTLayer.py:21-33)."""
    F = torch.nn.functional
    A = A.unsqueeze(0).permute(0, 3, 1, 2)

    def conv(name):
        return torch.sum(A * F.softmax(params[name], dim=1), dim=1)

    H = None
    for layer in range(num_layers):
        if layer == 0:
            H = torch.bmm(conv("layers.0.conv1.weight"), conv("layers.0.conv2.weight"))
        else:
            H = torch.stack([norm(H[c]) for c in range(num_channels)], dim=0)
            H = torch.bmm(H, conv(f"layers.{layer}.conv1.weight"))
    X_ = torch.cat([F.relu(gcn_conv(X, H[c], params["weight"])) for c in range(num_channels)], dim=1)
    X_ = F.relu(X_ @ params["linear1.weight"].t() + params["linear1.bias"])
    return X_[target_x] @ params["linear2.weight"].t() + params["linear2.bias"]
