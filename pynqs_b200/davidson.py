"""Block Davidson for the lowest eigenpairs of a real symmetric operator, in float64 torch on whatever device `diag` is on.

The operator enters only through `apply(V) -> H V`, so the solver runs on the device CSR product (`C_extension.csr_matmul`)
and, in the tests, on a host matrix.  Every step is a fixed sequence of torch calls; with a deterministic `apply` two runs
give the same bits.
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch
from torch import Tensor

# |theta - D_j| is kept at least this far from 0 in the preconditioner
_DENOM_MIN = 1.0e-8
# a new direction is dropped (deflation) when orthogonalisation leaves less than this fraction of its norm
_DROP = 1.0e-8


def _orthonormal_block(T: Tensor, V: Optional[Tensor]) -> Tensor:
    """Columns of T made orthonormal and orthogonal to the orthonormal V: two passes of block Gram-Schmidt against V, then
    QR inside the block.  Columns that (nearly) vanish on the way are dropped; a drop is followed by the whole sequence
    again on the remaining columns, so that no column is orthogonalised against a direction that QR made up."""
    T = T / T.norm(dim=0).clamp_min(torch.finfo(T.dtype).tiny)
    while T.shape[1] > 0:
        W = T
        if V is not None and V.shape[1] > 0:
            for _ in range(2):
                W = W - V @ (V.T @ W)
        Q, R = torch.linalg.qr(W)
        small = (R.diagonal().abs() <= _DROP).nonzero()
        if small.numel() == 0:
            if V is not None and V.shape[1] > 0:  # QR mixes the columns: one more pass keeps them orthogonal to V
                Q = torch.linalg.qr(Q - V @ (V.T @ Q)).Q
            return Q
        keep = torch.ones(T.shape[1], dtype=torch.bool, device=T.device)
        keep[int(small[0, 0])] = False
        T = T[:, keep]
    return T


def davidson(apply: Callable[[Tensor], Tensor], diag: Tensor, nroots: int = 1, guess: Optional[Tensor] = None, tol: float = 1e-8,
             max_iter: int = 200, max_subspace: Optional[int] = None) -> Tuple[Tensor, Tensor, dict]:
    """Lowest `nroots` eigenpairs of the symmetric operator `apply` (V [N, b] -> H V [N, b], float64).

    diag [N]: the diagonal of H, for the preconditioner t = r / (theta - D).  guess: [N] or [N, b] start vectors (default: unit
    vectors on the nroots lowest diagonal entries, ties broken by index); fewer than nroots columns are completed with those
    unit vectors.  A root has converged when ||H x - theta x||_2 <= tol with ||x|| = 1.  max_subspace (default
    max(8 nroots, 2 nroots + 16), at most N): when the basis would outgrow it, it restarts from the current Ritz vectors; a
    basis that may span the whole space never restarts.

    Returns (theta [nroots] ascending, X [N, nroots] orthonormal, info) with info = {"iterations", "products" (columns passed
    to apply), "residual_norms" (list of floats), "converged" (bool)}.  Running out of iterations is not an error:
    converged is False then."""
    diag = diag.reshape(-1).to(torch.float64)
    N, dev = diag.numel(), diag.device
    nroots = int(nroots)
    if not 1 <= nroots <= N:
        raise ValueError(f"nroots = {nroots} not in [1, N = {N}]")
    if max_subspace is None:
        max_subspace = max(8 * nroots, 2 * nroots + 16)
    max_subspace = min(int(max_subspace), N)
    if max_subspace < min(2 * nroots, N):
        raise ValueError(f"max_subspace = {max_subspace} must be at least 2 nroots = {2 * nroots} (or N)")
    order = torch.sort(diag, stable=True).indices[:nroots]
    units = torch.zeros(N, nroots, dtype=torch.float64, device=dev)
    units[order, torch.arange(nroots, device=dev)] = 1.0
    if guess is None:
        T = units
    else:
        g = guess.to(device=dev, dtype=torch.float64).reshape(N, -1)
        T = torch.cat([g, units[:, : max(nroots - g.shape[1], 0)]], dim=1)
    V = _orthonormal_block(T, None)
    if V.shape[1] < nroots:
        raise ValueError("the guess vectors are linearly dependent")
    AV = apply(V)
    products = V.shape[1]
    it = 0
    while True:
        G = V.T @ AV
        w, S = torch.linalg.eigh(0.5 * (G + G.T))
        theta, Y = w[:nroots], S[:, :nroots]
        X, AX = V @ Y, AV @ Y
        R = AX - X * theta
        rnorm = R.norm(dim=0)
        todo = rnorm > tol
        if not bool(todo.any()) or it >= max_iter:
            break
        it += 1
        denom = theta[todo] - diag[:, None]
        denom = torch.where(denom.abs() < _DENOM_MIN, torch.full_like(denom, _DENOM_MIN).copysign(denom), denom)
        T = R[:, todo] / denom
        if V.shape[1] + T.shape[1] > max_subspace and max_subspace < N:
            # thick restart: the Ritz vectors of the lowest min(2 nroots, room) values, H applied to them by linear algebra
            keep = max(nroots, min(2 * nroots, max_subspace - T.shape[1]))
            V, AV = V @ S[:, :keep], AV @ S[:, :keep]
        Q = _orthonormal_block(T, V)
        if Q.shape[1] == 0:
            break  # nothing new to add: the basis spans an invariant subspace to working precision
        V = torch.cat([V, Q], dim=1)
        AV = torch.cat([AV, apply(Q)], dim=1)
        products += Q.shape[1]
    info = {"iterations": it, "products": products, "residual_norms": [float(r) for r in rnorm.cpu()],
            "converged": not bool(todo.any())}
    return theta.clone(), X, info
