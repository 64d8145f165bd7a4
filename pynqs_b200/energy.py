"""Sample-space local energy (ElocMethod.SAMPLE_SPACE, vmc/energy/eloc.py:326-397) on the new ops.

`local_energy_reduced` is the REDUCE method (eloc.py:257-297) on compacted rows.

Two sample-space routes with identical results:
  * `local_energy_sample_space`  -- the one-pass kernels (scan of the string-grouped table copies -> H_ij on
    the hits -> reduce); nothing of size [n, M] is materialised, so 10^6 samples are a single call;
  * `local_energy_three_call`    -- the reference's sequence get_comb_hij_fused ->
    WavefunctionLUT.lookup -> scatter/divide/multiply/sum, chunked like vmc/energy/etot.py:76-146,
    kept so the unchanged reference Python keeps working on the new operators.
"""
from __future__ import annotations

from typing import Tuple

import torch
from torch import Tensor

from . import C_extension as ops
from .davidson import davidson
from .lut import WavefunctionLUT


def Func(func, x: Tensor, WF_LUT: "WavefunctionLUT | None" = None, use_unique: bool = False) -> Tensor:
    """psi of every row of x: table values where the LUT has the row, `func` (the ansatz) on the rest -- on the distinct
    rows only when use_unique.  Mirror of vmc/energy/flip.py:29-63 on the library's lookup + compaction
    (WavefunctionLUT.lookup) and its sort-based unique_onv instead of torch.unique(dim=0)."""
    batch = x.size(0)
    lut_idx = lut_not_idx = lut_value = None
    if WF_LUT is not None:
        lut_idx, lut_not_idx, lut_value = WF_LUT.lookup(x)
        x = x[lut_not_idx]
    if use_unique and x.size(0) > 0:
        unique_x, inverse = ops.unique_onv(x.contiguous())
        psi0 = torch.index_select(func(unique_x), 0, inverse)
    else:
        psi0 = func(x)
    if WF_LUT is None:
        return psi0
    psi = torch.empty(batch, dtype=psi0.dtype, device=psi0.device)
    psi[lut_idx] = lut_value.to(psi0.dtype)
    psi[lut_not_idx] = psi0
    return psi


def local_energy_sample_space(x: Tensor, h1e: Tensor, h2e: Tensor, WF_LUT: WavefunctionLUT, sorb: int, nele: int,
                              noa: int, nob: int, dtype=torch.double) -> Tuple[Tensor, Tensor, Tensor]:
    """Returns (eloc, sloc, psi_x) like _only_sample_space (eloc.py:508); sloc is zero (no spin-raising)."""
    eloc, psi0 = ops.eloc_sample_space(x, h1e, h2e, sorb, nele, noa, nob, WF_LUT.bra_key, WF_LUT.wf_value, WF_LUT.group_index)
    return eloc.to(dtype), torch.zeros_like(eloc).to(dtype), psi0.to(dtype)


def sample_space_hamiltonian(x: Tensor, h1e: Tensor, h2e: Tensor, WF_LUT: WavefunctionLUT, sorb: int, nele: int,
                             noa: int, nob: int) -> Tensor:
    """H[i, j] = <x_i|H|WF_LUT.bra_key[j]> as a float64 torch.sparse_csr_tensor of shape [n, N]: the connections that
    local_energy_sample_space sums over, so (H @ psi)[i] = eloc[i] * psi_x[i] with psi = WF_LUT.wf_value.  With x = the
    table itself it is the square sample-space Hamiltonian (variational energy psi^T H psi / psi^T psi, selected-CI
    diagonalisation, many products H psi without rescanning)."""
    N = WF_LUT.bra_key.size(0)
    crow, col, val = ops.sample_space_hamiltonian(x, h1e, h2e, sorb, nele, noa, nob, WF_LUT.bra_key,
                                                  WF_LUT.group_index if N > 0 else None)
    return torch.sparse_csr_tensor(crow, col, val, size=(x.size(0), N))


def sample_space_ground_state(WF_LUT: WavefunctionLUT, h1e: Tensor, h2e: Tensor, sorb: int, nele: int, noa: int, nob: int,
                              nroots: int = 1, *, H: "Tensor | None" = None, guess: "Tensor | None" = None, tol: float = 1e-8,
                              max_iter: int = 200) -> Tuple[Tensor, Tensor, dict]:
    """The lowest `nroots` eigenpairs of the square sample-space Hamiltonian over the determinants of WF_LUT.bra_key: the
    variational energies within the sample set and their CI coefficients.  Block Davidson (pynqs_b200.davidson) with
    H X = C_extension.csr_matmul on the device CSR matrix and the diagonal <x|H|x> as preconditioner.

    H: sample_space_hamiltonian(WF_LUT.bra_key, ...) (built when not given; pass it to reuse it).  guess: [N] or [N, b] start
    vectors, e.g. the real part of a VMC psi (default: unit vectors on the nroots lowest diagonal entries, ties broken by
    table row).  Returns (energies [nroots] ascending, electronic like eloc; coeffs [N, nroots] orthonormal, rows in the
    order of WF_LUT.bra_key; info of davidson: iterations, products, residual_norms, converged)."""
    keys = WF_LUT.bra_key
    N = keys.size(0)
    if H is None:
        H = sample_space_hamiltonian(keys, h1e, h2e, WF_LUT, sorb, nele, noa, nob)
    if H.layout != torch.sparse_csr or tuple(H.shape) != (N, N):
        raise ValueError(f"H must be a sparse CSR tensor of shape ({N}, {N})")
    crow, col, val = H.crow_indices(), H.col_indices(), H.values()
    # <x|H|x> from the 3-D form: one ket per bra, bit-identical to the CSR diagonal, nothing of size nnz
    diag = ops.get_hij_torch(keys, keys.view(N, 1, keys.size(1)), h1e, h2e, sorb, nele).view(N)
    return davidson(lambda V: ops.csr_matmul(crow, col, val, V, N), diag, nroots, guess=guess, tol=tol, max_iter=max_iter)


def local_energy_three_call(x: Tensor, h1e: Tensor, h2e: Tensor, WF_LUT: WavefunctionLUT, sorb: int, nele: int,
                            noa: int, nob: int, dtype=torch.double, batch: int = 4096) -> Tuple[Tensor, Tensor, Tensor]:
    """The reference's op sequence (eloc.py:369-397) in chunks of `batch` samples."""
    n = x.size(0)
    M = ops.get_Num_SinglesDoubles(sorb, noa, nob) + 1
    eloc = torch.empty(n, dtype=WF_LUT.dtype, device=x.device)
    psi_x = torch.empty(n, dtype=WF_LUT.dtype, device=x.device)
    for b in range(0, n, batch):
        xb = x[b : b + batch]
        comb_x, comb_hij = ops.get_comb_hij_fused(xb, h1e, h2e, sorb, nele, noa, nob)
        x1 = comb_x.reshape(-1, comb_x.size(2))
        psi_x1 = torch.zeros(xb.size(0), M, device=x.device, dtype=WF_LUT.dtype)
        idx, _, value = WF_LUT.lookup(x1)
        psi_x1.view(-1)[idx] = value
        real = torch.double if not WF_LUT.dtype.is_complex else torch.double
        comb_hij = comb_hij.to(real)
        eloc[b : b + batch] = ((psi_x1.T / psi_x1[..., 0]).T * comb_hij).sum(-1)
        psi_x[b : b + batch] = psi_x1[..., 0]
    return eloc.to(dtype), torch.zeros_like(eloc).to(dtype), psi_x.to(dtype)


def local_energy_reduced(x: Tensor, h1e: Tensor, h2e: Tensor, psi_of, sorb: int, nele: int, noa: int, nob: int,
                         dtype=torch.double, eps: float = 1.0e-12, batch: int = 65536, eps_sample: int = 0, seed=None,
                         draws=None) -> Tuple[Tensor, Tensor, Tensor]:
    """ElocMethod.REDUCE (eloc.py:204-323).  eps_sample = 0: only the connected determinants with |<x|H|x'>| >= eps enter
    E_loc.  eps_sample > 0 (the setting of the shipped inputs, main.py:149-159): the sub-eps rows are importance-sampled,
    eps_sample draws per sample from p ~ |H|, and enter with (count / eps_sample) * H / p (eloc.py:257-283); `seed` / `draws`
    as in get_comb_hij_sampled (`draws` [n, eps_sample] covers all of x, it is sliced per batch).  `psi_of(x_kept uint8 [K, 8L]) -> Tensor [K]` supplies the
    amplitudes (the reference's Func(ansatz, x, WF_LUT, use_unique)); a WavefunctionLUT may be passed instead,
    absent determinants then count as 0.  Returns (eloc, sloc, psi_x) like _reduce_psi."""
    M = ops.get_Num_SinglesDoubles(sorb, noa, nob) + 1
    if isinstance(psi_of, WavefunctionLUT):
        lut = psi_of

        def psi_of(xk: Tensor) -> Tensor:  # noqa: F811
            found, _, value = lut.lookup(xk)
            out = torch.zeros(xk.size(0), dtype=lut.dtype, device=xk.device)
            out[found] = value
            return out

    elocs, psis = [], []
    for b in range(0, x.size(0), batch):
        if eps_sample > 0:
            xk, hij, idx, offsets = ops.get_comb_hij_sampled(
                x[b : b + batch], h1e, h2e, sorb, nele, noa, nob, eps, eps_sample,
                seed=None if seed is None else int(seed) + b, draws=None if draws is None else draws[b : b + batch])
        else:
            xk, hij, idx, offsets = ops.get_comb_hij_reduced(x[b : b + batch], h1e, h2e, sorb, nele, noa, nob, eps)
        psi = psi_of(xk)
        psi = psi.to(torch.complex128 if psi.is_complex() else torch.float64)
        e, p0 = ops.reduce_eloc(psi, hij, idx, offsets, M)
        elocs.append(e)
        psis.append(p0)
    eloc = torch.cat(elocs) if elocs else torch.empty(0, dtype=dtype, device=x.device)
    psi_x = torch.cat(psis) if psis else torch.empty(0, dtype=dtype, device=x.device)
    return eloc.to(dtype), torch.zeros_like(eloc).to(dtype), psi_x.to(dtype)
