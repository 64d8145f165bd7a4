"""Lowest eigenpairs of the sample-space Hamiltonian: the CSR x block product (pynqs_csr_spmm / C_extension.csr_matmul), the
block Davidson solver (pynqs_b200.davidson) and energy.sample_space_ground_state.  The solver is checked on the host with a
host matrix standing in for the operator; the product and the whole chain on the GPU."""
import ctypes
import itertools

import numpy as np
import pytest
import scipy.linalg
import scipy.sparse
import scipy.sparse.linalg
import torch

from oracle import oracle as O
from pynqs_b200 import C_extension as ops
from pynqs_b200 import _lib
from pynqs_b200 import synthetic as S
from pynqs_b200.davidson import davidson
from pynqs_b200.energy import sample_space_ground_state, sample_space_hamiltonian
from pynqs_b200.lut import WavefunctionLUT

from util import fe2s2

DEV = "cuda:0"
gpu = pytest.mark.gpu

# lowest three eigenvalues of H over the Fe2S2 CI space (18 496 determinants, all pairs within two excitations), from
# scipy.sparse.linalg.eigsh(k=3, which="SA", tol=1e-12) on the host matrix built with oracle.hij
FE2S2_CI_LOWEST = [-114.3785426621286, -114.35772955847762, -114.34255940058875]


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def host_operator(H):
    Ht = torch.from_numpy(H)
    return (lambda V: Ht @ V), torch.from_numpy(np.ascontiguousarray(np.diag(H)))


def check_solution(H, theta, X, info, nroots, tol=1e-8, eig_tol=1e-10):
    want = np.linalg.eigh(H)[0][:nroots]
    theta, X = theta.numpy(), X.numpy()
    assert info["converged"]
    np.testing.assert_allclose(theta, want, rtol=0, atol=eig_tol)
    assert (np.diff(theta) >= 0).all()
    res = np.linalg.norm(H @ X - X * theta, axis=0)
    assert (res <= tol).all() and max(info["residual_norms"]) <= tol
    assert np.abs(X.T @ X - np.eye(nroots)).max() <= 1e-12


def sparse_symmetric(N, seed, per_row=6):
    rng = np.random.default_rng(seed)
    A = scipy.sparse.random(N, N, density=per_row / N, random_state=rng, data_rvs=lambda k: rng.uniform(-1, 1, k)).toarray()
    return 0.5 * (A + A.T) + np.diag(rng.uniform(0.0, 50.0, N))


# ---- the solver on the host ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("nroots", [1, 4])
def test_davidson_sparse_diagonally_dominant(nroots):
    H = sparse_symmetric(2000, seed=11)
    apply, diag = host_operator(H)
    theta, X, info = davidson(apply, diag, nroots)
    check_solution(H, theta, X, info, nroots)
    assert info["products"] >= info["iterations"]


def test_davidson_small_subspace_restarts():
    H = sparse_symmetric(2000, seed=12)
    apply, diag = host_operator(H)
    theta, X, info = davidson(apply, diag, 2, max_subspace=6)
    check_solution(H, theta, X, info, 2)


def test_davidson_degenerate_pairs():
    """Two copies of one block: every eigenvalue twice; nroots = 2 returns the lowest one twice, with two orthogonal vectors."""
    B = sparse_symmetric(300, seed=13)
    H = scipy.linalg.block_diag(B, B)
    apply, diag = host_operator(H)
    theta, X, info = davidson(apply, diag, 2)
    check_solution(H, theta, X, info, 2)
    lo = np.linalg.eigh(B)[0][0]
    np.testing.assert_allclose(theta.numpy(), [lo, lo], rtol=0, atol=1e-10)


def test_davidson_exact_eigenvector_guess():
    H = sparse_symmetric(500, seed=14)
    w, U = np.linalg.eigh(H)
    apply, diag = host_operator(H)
    theta, X, info = davidson(apply, diag, 1, guess=torch.from_numpy(U[:, 0].copy()))
    assert info["converged"] and info["iterations"] == 0
    assert abs(float(theta[0]) - w[0]) < 1e-10
    # two roots from a guess of which one column is exact: its correction vanishes, the other's does not
    g = np.stack([U[:, 0], np.ones(500)], axis=1)
    theta, X, info = davidson(apply, diag, 2, guess=torch.from_numpy(g))
    assert torch.isfinite(X).all() and torch.isfinite(theta).all()
    check_solution(H, theta, X, info, 2)


def test_davidson_whole_space_smaller_than_the_subspace():
    H = sparse_symmetric(10, seed=15, per_row=3)
    apply, diag = host_operator(H)
    theta, X, info = davidson(apply, diag, 3, max_subspace=40)
    check_solution(H, theta, X, info, 3)


def test_davidson_out_of_iterations_is_not_an_error():
    H = sparse_symmetric(2000, seed=16)
    apply, diag = host_operator(H)
    theta, X, info = davidson(apply, diag, 2, max_iter=1)
    assert info["converged"] is False and info["iterations"] == 1
    assert theta.shape == (2,) and X.shape == (2000, 2)
    with pytest.raises(ValueError):
        davidson(apply, diag, 0)
    with pytest.raises(ValueError):
        davidson(apply, diag, 3, max_subspace=4)


def full_ci_keys(sorb, noA, noB):
    half = sorb // 2
    a = [sum(1 << (2 * k) for k in c) for c in itertools.combinations(range(half), noA)]
    b = [sum(1 << (2 * k + 1) for k in c) for c in itertools.combinations(range(half), noB)]
    return np.array([x | y for x in a for y in b], dtype=np.uint64).view(np.uint8).reshape(-1, 8)


def test_davidson_full_ci_12_spin_orbitals():
    keys = full_ci_keys(12, 3, 3)
    assert keys.shape[0] == 400
    h1e, h2e = S.random_packed_integrals(12, seed=21, symmetric=True)
    H = O.hij(keys, keys, h1e, h2e, 12, 6)
    assert np.abs(H - H.T).max() < 1e-12
    apply, diag = host_operator(H)
    theta, X, info = davidson(apply, diag, 3)
    check_solution(H, theta, X, info, 3)


# ---- the C ABI's argument checks need no device ------------------------------------------------------------------------
def test_csr_spmm_bad_arguments_on_the_cpu():
    lib = _lib.load()
    p = _lib.vp(256)  # never dereferenced: the checks come first

    def call(n=10, N=10, k=2, ldx=2, ldy=2, crow=p, col=p, val=p, X=p, Y=p):
        return lib.pynqs_csr_spmm(crow, col, val, _lib.i64(n), _lib.i64(N), X, _lib.i64(ldx), int(k), Y, _lib.i64(ldy), _lib.vp(None))

    null = _lib.vp(None)
    for bad in (dict(n=-1), dict(N=-1), dict(k=0), dict(k=9, ldx=9, ldy=9), dict(ldx=1), dict(ldy=1), dict(crow=null),
                dict(Y=null), dict(col=null), dict(val=null), dict(X=null)):
        assert call(**bad) == _lib.EVALUE, bad
    assert b"csr_spmm" in lib.pynqs_last_error()
    assert call(n=0, crow=null, col=null, val=null, X=null, Y=null) == 0  # no rows: nothing to do, nothing launched
    with pytest.raises(NotImplementedError):
        ops.csr_matmul(torch.zeros(3, dtype=torch.int64), torch.zeros(0, dtype=torch.int64), torch.zeros(0, dtype=torch.float64),
                       torch.zeros(4, dtype=torch.float64), 4)


# ---- the product on the GPU ------------------------------------------------------------------------------------------
def host_product(crow, col, val, N, X):
    return scipy.sparse.csr_matrix((val, col, crow), shape=(crow.size - 1, N)) @ X


def check_product(crow_d, col_d, val_d, N, seed):
    """csr_matmul against scipy for real blocks of every width class, complex blocks, a column slice, and 1-D vectors;
    every result twice, bit for bit"""
    crow, col, val = crow_d.cpu().numpy(), col_d.cpu().numpy(), val_d.cpu().numpy()
    absH = scipy.sparse.csr_matrix((np.abs(val), col, crow), shape=(crow.size - 1, N))
    rng = np.random.default_rng(seed)

    def agree(X, Y):
        want = host_product(crow, col, val, N, X)
        scale = absH @ np.abs(X)
        assert Y.shape == want.shape and Y.dtype == want.dtype
        assert (np.abs(Y - want) <= 1e-13 * scale + 1e-300).all()

    for k in (1, 2, 3, 8, 13):
        X = rng.standard_normal((N, k))
        Xd = dev(X)
        Y = ops.csr_matmul(crow_d, col_d, val_d, Xd, N)
        agree(X, Y.cpu().numpy())
        assert Y.cpu().numpy().tobytes() == ops.csr_matmul(crow_d, col_d, val_d, Xd, N).cpu().numpy().tobytes()
    Z = rng.standard_normal((N, 3)) + 1j * rng.standard_normal((N, 3))
    Yc = ops.csr_matmul(crow_d, col_d, val_d, dev(Z), N)
    assert Yc.dtype == torch.complex128
    agree(Z, Yc.cpu().numpy())
    z = Z[:, 1].copy()
    yz = ops.csr_matmul(crow_d, col_d, val_d, dev(z), N)
    assert yz.shape == (crow.size - 1,)
    agree(z, yz.cpu().numpy())
    W = rng.standard_normal((N, 8))
    Ws = dev(W)[:, 2:5]  # rows 8 apart, a 3-column slice: passed through ld, not copied
    assert Ws.stride() == (8, 1)
    agree(W[:, 2:5], ops.csr_matmul(crow_d, col_d, val_d, Ws, N).cpu().numpy())
    v = W[:, 0].copy()
    yv = ops.csr_matmul(crow_d, col_d, val_d, dev(v), N)
    assert yv.shape == (crow.size - 1,)
    agree(v, yv.cpu().numpy())


@gpu
def test_csr_matmul_fe2s2_ci_space():
    _need_gpu()
    f = fe2s2()
    sorb, nele, noA, noB = f["sorb"], f["nele"], f["noA"], f["noB"]
    lut = WavefunctionLUT(dev(f["ci"]), dev(S.random_psi(f["ci"].shape[0], seed=3)), sorb, DEV, rank=0, world_size=1)
    h1e, h2e = dev(f["h1e"]), dev(f["h2e"])
    crow, col, val = ops.sample_space_hamiltonian(lut.bra_key, h1e, h2e, sorb, nele, noA, noB, lut.bra_key, lut.group_index)
    assert col.numel() > 2 * 10**7  # ~1 171 entries per row
    check_product(crow, col, val, 18496, seed=1)


@gpu
def test_csr_matmul_rectangular_with_empty_rows():
    _need_gpu()
    keys = full_ci_keys(12, 3, 3)[np.random.default_rng(80).permutation(400)]
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(12, seed=81, symmetric=True))
    lut = WavefunctionLUT(dev(keys[:150]), dev(S.random_psi(150, seed=82)), 12, DEV, rank=0, world_size=1)
    x = dev(keys[100:400])  # 50 samples in the table, 250 not
    crow, col, val = ops.sample_space_hamiltonian(x, h1e, h2e, 12, 6, 3, 3, lut.bra_key, lut.group_index)
    check_product(crow, col, val, 150, seed=2)
    # every third row emptied, the first and the last included: empty rows give 0
    c, k, v = crow.cpu().numpy(), col.cpu().numpy(), val.cpu().numpy()
    rows = np.repeat(np.arange(c.size - 1), np.diff(c))
    keep = rows % 3 != 0
    lens = np.bincount(rows[keep], minlength=c.size - 1)
    lens[-1] = 0
    keep &= rows != c.size - 2
    c2 = np.concatenate([[0], np.cumsum(lens)])
    assert (lens == 0).sum() > 90 and c2[-1] > 0
    check_product(dev(c2), dev(k[keep]), dev(v[keep]), 150, seed=4)


@gpu
def test_csr_matmul_long_rows():
    """Rows of more than 10 000 entries (one CTA per row) next to shorter ones (a warp or 8 lanes per row) in one matrix."""
    _need_gpu()
    sorb, noA, noB = 100, 25, 25
    seeds = S.random_onvs(2, sorb, noA, noB, seed=44)
    comb = O.comb(seeds, sorb, noA, noB).reshape(-1, 16)
    rng = np.random.default_rng(45)
    keys = np.unique(np.concatenate([seeds, comb[rng.permutation(comb.shape[0])[:30000]]]), axis=0)
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(sorb, seed=47, symmetric=False))
    lut = WavefunctionLUT(dev(keys), dev(S.random_psi(keys.shape[0], seed=46)), sorb, DEV, rank=0, world_size=1)
    x = dev(np.concatenate([seeds, keys[rng.permutation(keys.shape[0])[:3000]], seeds]))
    crow, col, val = ops.sample_space_hamiltonian(x, h1e, h2e, sorb, noA + noB, noA, noB, lut.bra_key, lut.group_index)
    lens = np.diff(crow.cpu().numpy())
    assert lens.max() > 10_000 and (lens <= 2048).any()
    check_product(crow, col, val, keys.shape[0], seed=3)


@gpu
def test_csr_matmul_empty_and_bad_inputs():
    _need_gpu()
    i64, f64 = torch.int64, torch.float64
    z = lambda *s, dtype=f64: torch.zeros(s, dtype=dtype, device=DEV)  # noqa: E731
    # n = 0
    assert ops.csr_matmul(z(1, dtype=i64), z(0, dtype=i64), z(0), z(7, 3), 7).shape == (0, 3)
    # N = 0 and nnz = 0: every row is empty
    l0 = _lib.launch_count()
    y = ops.csr_matmul(z(5, dtype=i64), z(0, dtype=i64), z(0), z(0, 2), 0)
    assert y.shape == (4, 2) and not y.any()
    y = ops.csr_matmul(z(5, dtype=i64), z(0, dtype=i64), z(0), z(9, dtype=torch.complex128), 9)
    assert y.shape == (4,) and y.dtype == torch.complex128 and not y.any()
    assert _lib.launch_count() == l0  # nothing to do, nothing launched
    crow, col, val = torch.tensor([0, 1, 1], device=DEV), torch.tensor([2], device=DEV), torch.tensor([3.0], device=DEV, dtype=f64)
    y = ops.csr_matmul(crow, col, val, torch.arange(4.0, device=DEV, dtype=f64), 4)
    assert y.tolist() == [6.0, 0.0]
    with pytest.raises(ValueError):
        ops.csr_matmul(crow, col, val, torch.arange(4.0, device=DEV), 4)  # float32
    with pytest.raises(ValueError):
        ops.csr_matmul(crow, col, val, torch.arange(5.0, device=DEV, dtype=f64), 4)  # wrong N
    with pytest.raises(ValueError):
        ops.csr_matmul(crow.int(), col, val, torch.arange(4.0, device=DEV, dtype=f64), 4)
    with pytest.raises(ValueError):
        ops.csr_matmul(crow, col, val.float(), torch.arange(4.0, device=DEV, dtype=f64), 4)
    with pytest.raises(ValueError):
        ops.csr_matmul(crow, col, val, z(4, 2, 2), 4)


# ---- the ground state ------------------------------------------------------------------------------------------------
@gpu
def test_fe2s2_ci_space_lowest_three():
    _need_gpu()
    f = fe2s2()
    sorb, nele, noA, noB = f["sorb"], f["nele"], f["noA"], f["noB"]
    lut = WavefunctionLUT(dev(f["ci"]), dev(S.random_psi(f["ci"].shape[0], seed=3)), sorb, DEV, rank=0, world_size=1)
    h1e, h2e = dev(f["h1e"]), dev(f["h2e"])
    H = sample_space_hamiltonian(lut.bra_key, h1e, h2e, lut, sorb, nele, noA, noB)
    e, C, info = sample_space_ground_state(lut, h1e, h2e, sorb, nele, noA, noB, nroots=3, H=H)
    assert info["converged"], info
    np.testing.assert_allclose(e.cpu().numpy(), FE2S2_CI_LOWEST, rtol=0, atol=1e-9)
    assert max(info["residual_norms"]) <= 1e-8
    # the residuals again, from the host matrix
    Hh = scipy.sparse.csr_matrix((H.values().cpu().numpy(), H.col_indices().cpu().numpy(), H.crow_indices().cpu().numpy()),
                                 shape=(18496, 18496))
    Ch = C.cpu().numpy()
    assert (np.linalg.norm(Hh @ Ch - Ch * e.cpu().numpy(), axis=0) <= 1e-8).all()
    assert np.abs(Ch.T @ Ch - np.eye(3)).max() <= 1e-12
    w, U = scipy.sparse.linalg.eigsh(Hh, k=3, which="SA", tol=1e-12)
    assert abs(U[:, np.argmin(w)] @ Ch[:, 0]) >= 1 - 1e-10
    # again, from scratch: the same bits
    e2, C2, _ = sample_space_ground_state(lut, h1e, h2e, sorb, nele, noA, noB, nroots=3)
    assert e2.cpu().numpy().tobytes() == e.cpu().numpy().tobytes()
    assert C2.cpu().numpy().tobytes() == Ch.tobytes()
    # a VMC-like guess (here: the solution, perturbed) converges to the same state
    g = C[:, 0] + 1e-3 * lut.wf_value
    e3, _, info3 = sample_space_ground_state(lut, h1e, h2e, sorb, nele, noA, noB, H=H, guess=g)
    assert info3["converged"] and abs(float(e3[0]) - FE2S2_CI_LOWEST[0]) < 1e-9


@gpu
def test_uniform_samples_as_their_own_table():
    _need_gpu()
    import bench

    f = fe2s2()
    sorb, nele, noA, noB = f["sorb"], f["nele"], f["noA"], f["noB"]
    keys = bench.make_table("uniform", 100_000)
    lut = WavefunctionLUT(dev(keys), dev(S.random_psi(keys.shape[0], seed=9)), sorb, DEV, rank=0, world_size=1)
    h1e, h2e = dev(f["h1e"]), dev(f["h2e"])
    H = sample_space_hamiltonian(lut.bra_key, h1e, h2e, lut, sorb, nele, noA, noB)
    e, C, info = sample_space_ground_state(lut, h1e, h2e, sorb, nele, noA, noB, nroots=2, H=H)
    assert info["converged"], info
    n = keys.shape[0]
    Hh = scipy.sparse.csr_matrix((H.values().cpu().numpy(), H.col_indices().cpu().numpy(), H.crow_indices().cpu().numpy()), shape=(n, n))
    w = np.sort(scipy.sparse.linalg.eigsh(Hh, k=2, which="SA", tol=1e-12)[0])
    np.testing.assert_allclose(e.cpu().numpy(), w, rtol=0, atol=1e-9)
