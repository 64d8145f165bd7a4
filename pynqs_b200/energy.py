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
                              max_iter: int = 200, spin_shift: float = 0.0, ss: "float | None" = None) -> Tuple[Tensor, Tensor, dict]:
    """The lowest `nroots` eigenpairs of the square sample-space Hamiltonian over the determinants of WF_LUT.bra_key: the
    variational energies within the sample set and their CI coefficients.  Block Davidson (pynqs_b200.davidson) with
    H X = C_extension.csr_matmul on the device CSR matrix and the diagonal <x|H|x> as preconditioner.

    H: sample_space_hamiltonian(WF_LUT.bra_key, ...) (built when not given; pass it to reuse it).  guess: [N] or [N, b] start
    vectors, e.g. the real part of a VMC psi (default: unit vectors on the nroots lowest diagonal entries, ties broken by
    table row).  Returns (energies [nroots] ascending, electronic like eloc; coeffs [N, nroots] orthonormal, rows in the
    order of WF_LUT.bra_key; info of davidson: iterations, products, residual_norms, converged).

    spin_shift > 0 targets a spin state, as PySCF's fix_spin_(shift, ss) does: the solver works on H + spin_shift S^2
    (ss = None: the lowest spins come first) or on H + spin_shift (S^2 - ss)^2 (the states with <S^2> = ss come first), with
    S^2 restricted to the sample set (C_extension.spin_square_matmul) and the exact diagonal of that operator as
    preconditioner.  The roots are then ordered by the penalised eigenvalues, `energies` are <c|H|c> of the converged
    vectors, and info["s2"] holds <c|S^2|c> of each root.  The penalty pins a spin only where the sample set is closed under
    spin exchanges (the CI space is; a random sample set is not, and its restricted S^2 has no exact spin eigenstates).
    The iterations grow with spin_shift, because the diagonal preconditioner does not see the penalty's spin-exchange
    couplings: take the smallest shift that lifts the other sectors above the wanted state.  spin_shift = 0 (the default)
    solves H alone."""
    keys = WF_LUT.bra_key
    N = keys.size(0)
    if spin_shift < 0 or (ss is not None and spin_shift == 0):
        raise ValueError(f"spin_shift = {spin_shift} must be >= 0, and > 0 when ss is given")
    if H is None:
        H = sample_space_hamiltonian(keys, h1e, h2e, WF_LUT, sorb, nele, noa, nob)
    if H.layout != torch.sparse_csr or tuple(H.shape) != (N, N):
        raise ValueError(f"H must be a sparse CSR tensor of shape ({N}, {N})")
    crow, col, val = H.crow_indices(), H.col_indices(), H.values()
    # <x|H|x> from the 3-D form: one ket per bra, bit-identical to the CSR diagonal, nothing of size nnz
    diag = ops.get_hij_torch(keys, keys.view(N, 1, keys.size(1)), h1e, h2e, sorb, nele).view(N)
    if spin_shift == 0:
        return davidson(lambda V: ops.csr_matmul(crow, col, val, V, N), diag, nroots, guess=guess, tol=tol, max_iter=max_iter)

    def h_apply(V: Tensor) -> Tensor:
        return ops.csr_matmul(crow, col, val, V, N)

    def s2_apply(V: Tensor) -> Tensor:
        return ops.spin_square_matmul(keys, sorb, keys, V, WF_LUT.group_index)

    d = _spin_diagonal(keys)  # every key is in its own table: the restricted S^2 has d on its diagonal
    if ss is None:
        def apply(V: Tensor) -> Tensor:
            return h_apply(V) + spin_shift * s2_apply(V)

        pdiag = diag + spin_shift * d
    else:
        def apply(V: Tensor) -> Tensor:
            W = s2_apply(V) - ss * V
            return h_apply(V) + spin_shift * (s2_apply(W) - ss * W)

        # diagonal of (S^2 - ss)^2: (d_i - ss)^2 + m_i, m_i = the in-table partners of row i, each an element +1;
        # S^2 applied to ones gives d_i + m_i
        m = s2_apply(torch.ones(N, dtype=torch.float64, device=keys.device)) - d
        pdiag = diag + spin_shift * ((d - ss) ** 2 + m)
    _, C, info = davidson(apply, pdiag, nroots, guess=guess, tol=tol, max_iter=max_iter)
    norm = (C * C).sum(0)
    info["s2"] = ((C * s2_apply(C)).sum(0) / norm).tolist()
    return (C * h_apply(C)).sum(0) / norm, C, info


def sample_space_pt2(WF_LUT: WavefunctionLUT, C: Tensor, energies: Tensor, h1e: Tensor, h2e: Tensor, sorb: int, nele: int, noa: int,
                     nob: int, *, max_bytes: int = 16 << 30) -> Tuple[Tensor, dict]:
    """The Epstein-Nesbet second-order correction of sample-space states, what selected CI (CIPSI, HCI) reports next to the
    variational energy as E_var + E_PT2:
        E_PT2[r] = (1 / sum_i C[i, r]^2) sum over a in X of (sum_i <key_i|H|a> C[i, r])^2 / (E[r] - <a|H|a>)
    with X the externals -- the distinct single and double excitations of the table's determinants (WF_LUT.bra_key, one
    (noa, nob) sector, no duplicates) that are not in the table.  <key_i|H|a> has the bits of get_comb_hij_fused, <a|H|a>
    those of get_hij_torch(a, a); both are electronic, like the energies of sample_space_ground_state, so
    `e, C, _ = sample_space_ground_state(...)` passes straight through.  A table that is the whole sector gives 0.

    C: float64 [N] or [N, k] (columns = states, rows in the order of WF_LUT.bra_key); energies: [k].  Returns (e_pt2 float64
    [k], info) with info["externals"] = |X|, info["pairs"] = the (row, external) pairs summed, info["passes"].  The externals
    are handled in passes of a hash partition each, as many as it takes to keep a pass's scratch within max_bytes (a memory
    limit; it changes the result only by rounding).  Deterministic: two calls with the same inputs and max_bytes give
    identical bits.  ValueError for a C of the wrong shape or dtype, energies of the wrong length, a zero column, a table
    with duplicate keys, non-float64 integrals or an empty table."""
    keys = WF_LUT.bra_key
    N = keys.size(0)
    if N == 0:
        raise ValueError("the table is empty")
    if C.dtype != torch.float64 or C.dim() not in (1, 2) or C.size(0) != N:
        raise ValueError(f"C must be float64 [N] or [N, k] with N = {N}, got {C.dtype} {tuple(C.shape)}")
    C2 = C.unsqueeze(1) if C.dim() == 1 else C
    k = C2.size(1)
    energies = torch.as_tensor(energies, dtype=torch.float64, device=keys.device).reshape(-1)
    if energies.numel() != k or k == 0:
        raise ValueError(f"energies must hold one value per column of C ({k}), got {energies.numel()}")
    if h1e.dtype != torch.float64 or h2e.dtype != torch.float64:
        raise ValueError("sample_space_pt2 needs float64 integrals")
    norm = (C2 * C2).sum(0)
    dup = (keys[1:] == keys[:-1]).all(1).any() if N > 1 else torch.zeros((), dtype=torch.bool, device=keys.device)
    zero, has_dup = torch.stack([(norm == 0).any(), dup]).tolist()
    if zero:
        raise ValueError("C has a column with sum c^2 = 0")
    if has_dup:
        raise ValueError("the table has duplicate keys")
    acc, info = ops.pt2_sums(keys, C2, energies, h1e, h2e, sorb, nele, noa, nob, WF_LUT.group_index, max_bytes=max_bytes)
    return acc / norm, info


def _spin_diagonal(x: Tensor) -> Tensor:
    """<x|S^2|x> = |B| + Sz (Sz + 1) of every ONV row of x (uint8 [n, 8L]), float64 [n]: B = the beta-only orbitals,
    Sz = (n_alpha - n_beta) / 2 (alpha on the even bits, beta on the odd ones)."""
    pc = torch.tensor([bin(v).count("1") for v in range(256)], dtype=torch.int64, device=x.device)
    b = x.long()
    alpha, beta = b & 0x55, (b >> 1) & 0x55  # the orbitals of each byte, alpha- and beta-occupied
    na, nb, nB = pc[alpha].sum(1), pc[beta].sum(1), pc[beta & ~alpha].sum(1)
    sz2 = (na - nb).to(torch.float64)
    return nB.to(torch.float64) + 0.25 * sz2 * (sz2 + 2.0)


def local_spin_square(x: Tensor, WF_LUT: WavefunctionLUT, sorb: int) -> Tuple[Tensor, Tensor]:
    """The local spin of every sample, S^2_loc(x) = (S^2 psi)(x) / psi(x) with psi = WF_LUT.wf_value over the table (the
    sample-space convention of local_energy_sample_space: spin exchanges of x that are not in the table count as psi = 0).
    Returns (s2loc [n], psi_x [n]) in psi's dtype (float64 or complex128); the |psi|^2-weighted mean of s2loc over the table
    is <S^2> of psi (spin_square).  A sample that is not in the table gets psi_x = 0 and s2loc = NaN, as
    local_energy_sample_space gives it psi_x = 0 and E_loc = 0/0 = NaN; so does a sample whose table value is 0."""
    N = WF_LUT.bra_key.size(0)
    s2psi = ops.spin_square_matmul(x, sorb, WF_LUT.bra_key, WF_LUT.wf_value, WF_LUT.group_index if N > 0 else None)
    found, _, value = WF_LUT.lookup(x)
    psi_x = torch.zeros_like(s2psi)
    psi_x[found] = value
    nan = complex(float("nan"), float("nan")) if s2psi.is_complex() else float("nan")
    return torch.where(psi_x == 0, torch.full_like(s2psi, nan), s2psi / psi_x), psi_x


def spin_square(WF_LUT: WavefunctionLUT, C: Tensor, sorb: int) -> Tensor:
    """<S^2> = Re(c^H S^2 c) / (c^H c) of every column c of C (float64 or complex128, [N] or [N, k], rows in the order of
    WF_LUT.bra_key: Davidson coefficients, or WF_LUT.wf_value), with S^2 restricted to the table.  Returns float64 [k]
    ([1] for a 1-D C)."""
    keys = WF_LUT.bra_key
    C = C.unsqueeze(1) if C.dim() == 1 else C
    S2C = ops.spin_square_matmul(keys, sorb, keys, C, WF_LUT.group_index)
    return (C.conj() * S2C).sum(0).real / (C.conj() * C).sum(0).real


def make_rdm1s(WF_LUT: WavefunctionLUT, C: Tensor, sorb: int, H: Tensor) -> Tuple[Tensor, Tensor]:
    """The one-body reduced density matrices (dm1a, dm1b) of the state C over the table, dm1s[p, q] = <c|a+_qs a_ps|c> / <c|c>
    (PySCF's make_rdm1s): see make_rdm12s for the arguments and conventions.  Skips the two-body work; its dm1 has the bits
    of make_rdm12s's.  The natural occupations are eigvalsh(dm1a + dm1b)."""
    dm1, _ = _make_rdm(WF_LUT, C, sorb, H, False)
    return dm1[0], dm1[1]


def make_rdm12s(WF_LUT: WavefunctionLUT, C: Tensor, sorb: int, H: Tensor) -> Tuple[Tuple[Tensor, Tensor], Tuple[Tensor, Tensor, Tensor]]:
    """The one- and two-body reduced density matrices of the state C over the table, in PySCF's make_rdm12s conventions:
    ((dm1a, dm1b), (dm2aa, dm2ab, dm2bb)) with dm1s[p, q] = <c|a+_qs a_ps|c> / <c|c> ([norb, norb], norb = sorb / 2) and
    dm2st[p, q, r, s] = <c|a+_ps a+_rt a_st a_qs|c> / <c|c> ([norb]^4).  Orbital p has alpha at bit 2p and beta at 2p + 1,
    and the sign is get_hij_torch's.  Sums run over pairs of table rows only -- the sample-space convention of
    local_energy_sample_space and spin_square: a determinant outside the table counts as c = 0 --, so with H the energy
    sum h (dm1a + dm1b) + 1/2 sum eri dm2aa + sum eri dm2ab + 1/2 sum eri dm2bb equals Re(c^H H c) / c^H c.  The natural
    occupations are eigvalsh(dm1a + dm1b).

    C: float64 or complex128 [N], rows in the order of WF_LUT.bra_key (a CI root of sample_space_ground_state, or
    WF_LUT.wf_value); the result has C's dtype (complex dm1 is Hermitian).  H: the square
    sample_space_hamiltonian(WF_LUT.bra_key, ...) of the same table, of which only the structure is read.  ValueError when
    H is not (N, N) CSR, C has the wrong shape or dtype, sum |c|^2 = 0, or the table has duplicate keys.  Deterministic
    (identical bits on every call); two host synchronisations."""
    dm1, dm2 = _make_rdm(WF_LUT, C, sorb, H, True)
    return (dm1[0], dm1[1]), (dm2[0], dm2[1], dm2[2])


def _make_rdm(WF_LUT: WavefunctionLUT, C: Tensor, sorb: int, H: Tensor, two_body: bool) -> Tuple[Tensor, "Tensor | None"]:
    keys = WF_LUT.bra_key
    N = keys.size(0)
    if H.layout != torch.sparse_csr or tuple(H.shape) != (N, N):
        raise ValueError(f"H must be a sparse CSR tensor of shape ({N}, {N})")
    if C.dtype not in (torch.float64, torch.complex128) or C.shape != (N,):
        raise ValueError(f"C must be float64 or complex128 of shape ({N},), got {C.dtype} {tuple(C.shape)}")
    w = torch.view_as_real(C).square().sum(1) if C.is_complex() else C * C  # |c_i|^2
    norm = w.sum()
    dup = (keys[1:] == keys[:-1]).all(1).any() if N > 1 else torch.zeros((), dtype=torch.bool, device=keys.device)
    zero, has_dup = torch.stack([norm == 0, dup]).tolist()
    if zero:
        raise ValueError("C has sum |c|^2 = 0")
    if has_dup:
        raise ValueError("the table has duplicate keys")
    dm1, dm2 = ops.rdm_offdiag(H.crow_indices(), H.col_indices(), keys, C.contiguous(), sorb, two_body)
    # the diagonal pairs: |c_i|^2 times occupation products, as dense products over the occupations Occ [N, 2, norb]
    norb = sorb // 2
    bits = (keys.unsqueeze(2) >> torch.arange(8, device=keys.device, dtype=torch.uint8)) & 1
    occ = bits.view(N, -1)[:, :sorb].view(N, norb, 2).permute(0, 2, 1).contiguous().to(torch.float64)
    ar = torch.arange(norb, device=keys.device)
    dm1[:, ar, ar] += (w @ occ.view(N, 2 * norb)).view(2, norb).to(dm1.dtype)
    if two_body:
        wocc = occ * w.view(N, 1, 1)
        for blk, (s, t) in enumerate(((0, 0), (0, 1), (1, 1))):
            G = (wocc[:, s].T @ occ[:, t]).to(dm2.dtype)  # sum |c_i|^2 n_ps n_rt
            if s == t:
                G.fill_diagonal_(0)  # a+_p a+_p = 0
                dm2[blk, ar[:, None], ar[None, :], ar[None, :], ar[:, None]] -= G  # <a+_p a+_r a_p a_r> = -n_p n_r
            dm2[blk, ar[:, None], ar[:, None], ar[None, :], ar[None, :]] += G
        dm2 /= norm
    dm1 /= norm
    return dm1, dm2


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
