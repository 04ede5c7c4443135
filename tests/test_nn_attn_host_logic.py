"""Host-side pieces of the fused Q|K'|V' projection + chain attention (gnnlm_linear_f16f8_nn_attn): the head-interleaved weight
order and the row windows.  CPU only."""
import numpy as np
import pytest
import torch


@pytest.mark.parametrize("H", [2, 4, 8])
def test_head_interleave_reproduces_qkv_columns(H):
    """Permuted rows give the permuted columns of the same product: N-tile h (256 columns) = [Q_h | K'_h], tile H + j = V' of
    heads 2j, 2j + 1."""
    from gnnlm_b200.hgt import head_interleave
    dk, K = 128, 64
    d = H * dk
    g = torch.Generator().manual_seed(H)
    W = torch.randn(3 * d, K, generator=g, dtype=torch.float64)
    b = torch.randn(3 * d, generator=g, dtype=torch.float64)
    x = torch.randn(5, K, generator=g, dtype=torch.float64)
    perm = head_interleave(H, dk)
    assert sorted(perm.tolist()) == list(range(3 * d))
    y = x @ W.T + b
    yp = x @ W[perm].T + b[perm]
    torch.testing.assert_close(yp, y[:, perm], rtol=0, atol=1e-12)
    q, k, v = y[:, :d], y[:, d:2 * d], y[:, 2 * d:]
    for h in range(H):
        tile = yp[:, 256 * h:256 * (h + 1)]
        torch.testing.assert_close(tile[:, :dk], q[:, h * dk:(h + 1) * dk], rtol=0, atol=1e-12)
        torch.testing.assert_close(tile[:, dk:], k[:, h * dk:(h + 1) * dk], rtol=0, atol=1e-12)
    for j in range(H // 2):
        tile = yp[:, 2 * d + 256 * j:2 * d + 256 * (j + 1)]
        torch.testing.assert_close(tile, v[:, 256 * j:256 * (j + 1)], rtol=0, atol=1e-12)


@pytest.mark.parametrize("w", [1, 3, 5, 7])
@pytest.mark.parametrize("M", [1, 127, 128, 129, 292040])
def test_window_plan_owns_every_row_once_with_its_chain(w, M):
    """Every row is owned by exactly one window, and every id within w - 1 of an owned row (any chain neighbour in a cluster of
    at most w contiguous ids) is one of the 128 rows that window loads."""
    from gnnlm_b200.ops import nn_window_plan
    h, S, n_win = nn_window_plan(M, w)
    assert S == 128 - 2 * h and S > 0
    owners = np.zeros(M, dtype=np.int64)
    for j in range(n_win):
        owners[j * S:min(j * S + S, M)] += 1
    assert (owners == 1).all()
    g = np.arange(M)
    j = g // S
    lo, hi = j * S - h, j * S - h + 128
    for off in range(-h, h + 1):
        m = g + off
        inside = (m >= 0) & (m < M)
        assert ((m[inside] >= lo[inside]) & (m[inside] < hi[inside])).all()
    assert n_win == 0 or (n_win - 1) * S < M
