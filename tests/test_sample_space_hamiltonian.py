"""The sample-space Hamiltonian as a CSR matrix (pynqs_hamiltonian_count / _emit): against the dense get_hij_torch(bra, key)
(values bit for bit, the pattern = the entries eloc_sample_space sums over), against eloc_sample_space through
(H psi)[i] = eloc[i] * psi0[i], on every scan route and the reference's route."""
import ctypes
import itertools

import numpy as np
import pytest
import torch

from oracle import oracle as O
from pynqs_b200 import C_extension as ops
from pynqs_b200 import _lib
from pynqs_b200 import synthetic as S
from pynqs_b200.energy import sample_space_hamiltonian
from pynqs_b200.lut import WavefunctionLUT

from util import fe2s2

DEV = "cuda:0"
gpu = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.fixture(autouse=True)
def _default_tuning():
    _lib.set_tuning()
    yield
    _lib.set_tuning()


@pytest.fixture(params=["folded", "full_keys", "block", "block_whole_tiles", "block_4_parts", "full_keys_tiles"])
def scan_route(request):
    """One-word ONVs are scanned through folded 32-bit strings; the knob full_keys forces the full-key
    route that multi-word ONVs (and tables of 2^30 keys or more) take; "block" sends every call, however small, through
    the grouping pass and the block kernel (samples sharing a beta string walk their groups together), with tiles from
    4 samples on.  All must give the same numbers."""
    if request.param == "full_keys":
        _lib.set_tuning("full_keys", 1)
    elif request.param == "full_keys_tiles":
        _lib.set_tuning("full_keys", 1)
        _lib.set_tuning("eval_tiles", 2)
    elif request.param.startswith("block"):
        _lib.set_tuning("block_min_samples", 1)
        _lib.set_tuning("block_min_group", 4)
        _lib.set_tuning("eval_tiles", 2)  # ... and the evaluation kernel that takes 32 samples per warp
        # the alpha-beta groups of a tile walked by one warp, or split over 4 ("block": the kernel's own choice, 2 for small calls)
        if request.param != "block":
            _lib.set_tuning("block_parts", 1 if request.param == "block_whole_tiles" else 4)
    return request.param


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")


def csr(x, h1e, h2e, lut, sorb, nele, noA, noB):
    """(crow, col, val) on the host"""
    crow, col, val = ops.sample_space_hamiltonian(x, h1e, h2e, sorb, nele, noA, noB, lut.bra_key, lut.group_index)
    return crow.cpu().numpy(), col.cpu().numpy(), val.cpu().numpy()


def check_structure(crow, col, N):
    assert crow[0] == 0 and (np.diff(crow) >= 0).all() and crow[-1] == col.size
    assert ((col >= 0) & (col < N)).all()
    starts = np.zeros(col.size, dtype=bool)
    starts[crow[:-1][crow[:-1] < col.size]] = True
    asc = np.diff(col) > 0
    assert (asc | starts[1:]).all(), "columns must ascend strictly within a row"


def check_against_dense(crow, col, val, H):
    """values bit-identical at the stored positions, the dense matrix zero everywhere else"""
    rows = np.repeat(np.arange(crow.size - 1), np.diff(crow))
    np.testing.assert_array_equal(val.view(np.uint64), H[rows, col].view(np.uint64))
    rest = H.copy()
    rest[rows, col] = 0.0
    assert not rest.any()


def matvec(crow, col, val, v):
    """(H v) for real or complex v, as two real products"""
    rows = np.repeat(np.arange(crow.size - 1), np.diff(crow))
    out = np.zeros(crow.size - 1, dtype=v.dtype)
    np.add.at(out, rows, val * v[col])
    return out


def check_eloc_identity(x, h1e, h2e, lut, sorb, nele, noA, noB, crow, col, val, rtol=1e-12):
    eloc, psi0 = ops.eloc_sample_space(x, h1e, h2e, sorb, nele, noA, noB, lut.bra_key, lut.wf_value, lut.group_index)
    psi = lut.wf_value.cpu().numpy()
    Hpsi = matvec(crow, col, val, psi)
    want = eloc.cpu().numpy() * psi0.cpu().numpy()
    np.testing.assert_allclose(Hpsi.real, want.real, rtol=rtol, atol=rtol * np.abs(want).max())
    if np.iscomplexobj(psi):
        np.testing.assert_allclose(Hpsi.imag, want.imag, rtol=rtol, atol=rtol * np.abs(want).max())
    return eloc, psi0


def excitation_level(a, b):
    """number of electrons moved between two ONV tables (uint8 [*, 8L]), as a matrix"""
    bits_a = np.unpackbits(a, axis=1, bitorder="little").astype(np.int16)
    bits_b = np.unpackbits(b, axis=1, bitorder="little").astype(np.int16)
    return (bits_a[:, None, :] != bits_b[None, :, :]).sum(-1) // 2


# ---- host side --------------------------------------------------------------------------------------------------
def test_scratch_bytes_on_the_cpu():
    """pynqs_hamiltonian_scratch_bytes needs no GPU: it grows with n and by 16 bytes per entry, and refuses bad input."""
    lib = _lib.load()
    nb = ctypes.c_int64()

    def size(n, nnz, sorb=40, noA=15, noB=15):
        rc = lib.pynqs_hamiltonian_scratch_bytes(_lib.i64(n), _lib.i64(nnz), sorb, noA, noB, ctypes.byref(nb))
        return rc, nb.value

    rc, s0 = size(1000, 0)
    assert rc == 0 and s0 > 0
    rc, s1 = size(1000, 10_000)
    assert rc == 0 and s1 - s0 >= 16 * 10_000 and s1 - s0 < 16 * 10_000 + 512
    assert size(2000, 0)[1] > s0
    el = ctypes.c_int64()
    assert lib.pynqs_eloc_scratch_bytes(_lib.i64(1000), 40, 15, 15, 0, ctypes.byref(el)) == 0 and s0 > el.value
    assert size(1000, 0, sorb=100, noA=25, noB=25)[0] == 0
    assert size(-1, 0)[0] == _lib.EVALUE
    assert size(10, -5)[0] == _lib.EVALUE
    assert size(10, 0, sorb=41)[0] == _lib.EVALUE


def test_cpu_tensors_raise():
    keys = torch.from_numpy(S.random_onvs(10, 12, 3, 3, seed=1))
    h1e, h2e = (torch.from_numpy(a) for a in S.random_packed_integrals(12, seed=2, symmetric=True))
    with pytest.raises(NotImplementedError):
        ops.sample_space_hamiltonian(keys, h1e, h2e, 12, 6, 3, 3, keys)
    lut = WavefunctionLUT(keys, torch.from_numpy(S.random_psi(10, seed=3)), 12, rank=0, world_size=1)
    with pytest.raises(NotImplementedError):
        sample_space_hamiltonian(keys, h1e, h2e, lut, 12, 6, 3, 3)


# ---- 1. full space, H6 shape ----------------------------------------------------------------------------------------
@gpu
def test_full_space_matches_dense_and_the_spectrum(scan_route):
    _need_gpu()
    keys = S.random_onvs(400, 12, 3, 3, seed=51)
    h1e_np, h2e_np = S.random_packed_integrals(12, seed=52, symmetric=True)
    psi = S.random_psi(400, seed=53)
    h1e, h2e = dev(h1e_np), dev(h2e_np)
    lut = WavefunctionLUT(dev(keys), dev(psi), 12, DEV, rank=0, world_size=1)
    skeys = lut.bra_key.cpu().numpy()
    crow, col, val = csr(lut.bra_key, h1e, h2e, lut, 12, 6, 3, 3)
    check_structure(crow, col, 400)
    H = ops.get_hij_torch(lut.bra_key, lut.bra_key, h1e, h2e, 12, 6).cpu().numpy()
    check_against_dense(crow, col, val, H)
    # the pattern: every pair within two excitations, the diagonal included
    rows = np.repeat(np.arange(400), np.diff(crow))
    pat = np.zeros((400, 400), dtype=bool)
    pat[rows, col] = True
    np.testing.assert_array_equal(pat, excitation_level(skeys, skeys) <= 2)
    D = np.zeros((400, 400))
    D[rows, col] = val
    np.testing.assert_array_equal(D, D.T)
    # variational energy from the sparse product, and the lowest eigenvalue against the oracle's dense H
    Hs = sample_space_hamiltonian(lut.bra_key, h1e, h2e, lut, 12, 6, 3, 3)
    assert Hs.layout == torch.sparse_csr and tuple(Hs.shape) == (400, 400)
    p = lut.wf_value.view(-1, 1)
    e_sparse = float((p.T @ torch.sparse.mm(Hs, p)).item() / (p.T @ p).item())
    q = p.cpu().numpy().reshape(-1)
    e_dense = float(q @ H @ q / (q @ q))
    assert abs(e_sparse - e_dense) < 1e-12
    import scipy.sparse
    import scipy.sparse.linalg

    M = scipy.sparse.csr_matrix((val, col, crow), shape=(400, 400))
    lo = scipy.sparse.linalg.eigsh(M, k=1, which="SA", tol=1e-14)[0][0]
    ref = np.linalg.eigvalsh(O.hij(skeys, skeys, h1e_np, h2e_np, 12, 6))[0]
    assert abs(lo - ref) < 1e-10
    # every route and tuning gives the same bytes
    _lib.set_tuning()
    base = csr(lut.bra_key, h1e, h2e, lut, 12, 6, 3, 3)
    for a, b in zip(base, (crow, col, val)):
        assert a.tobytes() == b.tobytes()


# ---- 2. Fe2S2 ci_space table -----------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("cplx", [False, True])
def test_fe2s2_ci_space(cplx, scan_route):
    _need_gpu()
    f = fe2s2()
    sorb, nele, noA, noB = f["sorb"], f["nele"], f["noA"], f["noB"]
    psi = S.random_psi(f["ci"].shape[0], seed=3, complex_=cplx)
    lut = WavefunctionLUT(dev(f["ci"]), dev(psi), sorb, DEV, rank=0, world_size=1)
    assert lut.bra_key.size(0) == 18496
    x = dev(f["ci"][100:164])
    h1e, h2e = dev(f["h1e"]), dev(f["h2e"])
    crow, col, val = csr(x, h1e, h2e, lut, sorb, nele, noA, noB)
    check_structure(crow, col, 18496)
    check_against_dense(crow, col, val, ops.get_hij_torch(x, lut.bra_key, h1e, h2e, sorb, nele).cpu().numpy())
    check_eloc_identity(x, h1e, h2e, lut, sorb, nele, noA, noB, crow, col, val)


# ---- 3. rectangular: samples missing from the table ------------------------------------------------------------------
@gpu
def test_rectangular_samples_missing_from_the_table(scan_route):
    _need_gpu()
    keys = S.random_onvs(300, 12, 3, 3, seed=80)
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(12, seed=81, symmetric=True))
    lut = WavefunctionLUT(dev(keys[:200]), dev(S.random_psi(200, seed=82)), 12, DEV, rank=0, world_size=1)
    x = dev(keys[190:210])
    crow, col, val = csr(x, h1e, h2e, lut, 12, 6, 3, 3)
    check_structure(crow, col, 200)
    check_against_dense(crow, col, val, ops.get_hij_torch(x, lut.bra_key, h1e, h2e, 12, 6).cpu().numpy())
    skeys = lut.bra_key.cpu().numpy()
    for i in range(20):
        cols = col[crow[i] : crow[i + 1]]
        diag = [j for j in cols if (skeys[j] == keys[190 + i]).all()]
        assert len(diag) == (1 if i < 10 else 0)
    Hs = sample_space_hamiltonian(x, h1e, h2e, lut, 12, 6, 3, 3)
    assert tuple(Hs.shape) == (20, 200)


# ---- 4. the reference's route ----------------------------------------------------------------------------------------
@gpu
def test_hit_queue_overflow_takes_the_reference_route(scan_route):
    _need_gpu()
    sorb, noA, noB, nele = 40, 15, 15, 30
    a = np.array([sum(1 << (2 * k) for k in c) for c in itertools.combinations(range(20), 15)], dtype=np.uint64)
    b = np.array([sum(1 << (2 * k + 1) for k in c) for c in (range(15), list(range(14)) + [17], list(range(13)) + [15, 19])], dtype=np.uint64)
    keys = (a[:, None] | b[None, :]).reshape(-1).view(np.uint8).reshape(-1, 8)
    keys = keys[np.random.default_rng(3).permutation(keys.shape[0])]
    psi = S.random_psi(keys.shape[0], seed=4)
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(sorb, seed=7, symmetric=True))
    lut = WavefunctionLUT(dev(keys), dev(psi), sorb, DEV, rank=0, world_size=1)
    x = dev(keys[:40])
    crow, col, val = csr(x, h1e, h2e, lut, sorb, nele, noA, noB)
    check_structure(crow, col, keys.shape[0])
    assert np.diff(crow).max() > 512  # more hits than a scan queue takes
    check_against_dense(crow, col, val, ops.get_hij_torch(x, lut.bra_key, h1e, h2e, sorb, nele).cpu().numpy())
    check_eloc_identity(x, h1e, h2e, lut, sorb, nele, noA, noB, crow, col, val)


@gpu
@pytest.mark.parametrize("route", ["default", "block"])
@pytest.mark.parametrize("sorb,noA,noB", [(40, 15, 15), (100, 3, 3)])
def test_table_with_duplicate_keys(sorb, noA, noB, route):
    """Columns are the rows the classic binary search lands on; (H psi)[i] = eloc[i] psi0[i] with the copies' different psi."""
    _need_gpu()
    if route == "block":
        _lib.set_tuning("block_min_samples", 1)
        _lib.set_tuning("block_min_group", 4)
        _lib.set_tuning("eval_tiles", 2)
    seeds = S.random_onvs(3, sorb, noA, noB, seed=61)
    comb = O.comb(seeds, sorb, noA, noB).reshape(-1, seeds.shape[1])
    rng = np.random.default_rng(62)
    keys = np.unique(np.concatenate([seeds, comb[rng.permutation(comb.shape[0])[:1500]]]), axis=0)
    keys = np.concatenate([keys, keys[::7], keys[::31]])
    psi = S.random_psi(keys.shape[0], seed=63)
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(sorb, seed=7, symmetric=True))
    lut = WavefunctionLUT(dev(keys), dev(psi), sorb, DEV, rank=0, world_size=1)
    x = dev(np.concatenate([seeds, keys[:9]]))
    nele = noA + noB
    crow, col, val = csr(x, h1e, h2e, lut, sorb, nele, noA, noB)
    check_structure(crow, col, keys.shape[0])
    # columns: the rows the classic search lands on for the connected keys; values: the dense matrix there
    H = ops.get_hij_torch(x, lut.bra_key, h1e, h2e, sorb, nele).cpu().numpy()
    idx, _ = ops.wavefunction_lut(lut.bra_key, lut.bra_key, sorb, hash_index=False)
    landing = idx.cpu().numpy()
    assert (landing != np.arange(keys.shape[0])).any()  # some copies are never landed on
    lvl = excitation_level(x.cpu().numpy(), lut.bra_key.cpu().numpy())
    for i in range(H.shape[0]):
        np.testing.assert_array_equal(col[crow[i] : crow[i + 1]], np.unique(landing[lvl[i] <= 2]))
    rows = np.repeat(np.arange(H.shape[0]), np.diff(crow))
    np.testing.assert_array_equal(val.view(np.uint64), H[rows, col].view(np.uint64))
    check_eloc_identity(x, h1e, h2e, lut, sorb, nele, noA, noB, crow, col, val)


# ---- 5. multi-word ONVs and long rows --------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("sorb,noA,noB,nkeys", [(100, 3, 3, 4000), (132, 3, 2, 3000), (192, 4, 4, 3000)])
def test_multiword_onvs(sorb, noA, noB, nkeys):
    _need_gpu()
    seeds = S.random_onvs(3, sorb, noA, noB, seed=sorb)
    comb = O.comb(seeds, sorb, noA, noB).reshape(-1, seeds.shape[1])
    rng = np.random.default_rng(1)
    keys = np.unique(np.concatenate([seeds, comb[rng.permutation(comb.shape[0])[: nkeys - 3]]]), axis=0)
    psi = S.random_psi(keys.shape[0], seed=2, complex_=(sorb == 132))
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(sorb, seed=3, symmetric=False))
    lut = WavefunctionLUT(dev(keys), dev(psi), sorb, DEV, rank=0, world_size=1)
    x = dev(np.concatenate([seeds, keys[:5]]))
    crow, col, val = csr(x, h1e, h2e, lut, sorb, noA + noB, noA, noB)
    check_structure(crow, col, keys.shape[0])
    check_against_dense(crow, col, val, ops.get_hij_torch(x, lut.bra_key, h1e, h2e, sorb, noA + noB).cpu().numpy())
    check_eloc_identity(x, h1e, h2e, lut, sorb, noA + noB, noA, noB, crow, col, val)


@gpu
def test_dense_24_orbital_space_full_rows(scan_route):
    """Full 24-spin-orbital space (6a6b, 853 776 keys): every connected determinant is in the table, so every row holds
    x itself and all nsd = 1818 excitations."""
    _need_gpu()
    sorb, noA, noB, nele = 24, 6, 6, 12
    strings = [sum(1 << (2 * k) for k in c) for c in itertools.combinations(range(12), 6)]
    a = np.array(strings, dtype=np.uint64)
    keys = (a[:, None] | (a[None, :] << np.uint64(1))).reshape(-1).view(np.uint8).reshape(-1, 8)
    keys = keys[np.random.default_rng(5).permutation(keys.shape[0])]
    psi = S.random_psi(keys.shape[0], seed=6)
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(sorb, seed=8, symmetric=True))
    lut = WavefunctionLUT(dev(keys), dev(psi), sorb, DEV, rank=0, world_size=1)
    x = dev(keys[:48])
    crow, col, val = csr(x, h1e, h2e, lut, sorb, nele, noA, noB)
    check_structure(crow, col, keys.shape[0])
    assert (np.diff(crow) == ops.get_Num_SinglesDoubles(sorb, noA, noB) + 1).all()  # 1819
    check_against_dense(crow, col, val, ops.get_hij_torch(x, lut.bra_key, h1e, h2e, sorb, nele).cpu().numpy())
    check_eloc_identity(x, h1e, h2e, lut, sorb, nele, noA, noB, crow, col, val)


@gpu
def test_h50_shape_long_rows():
    _need_gpu()
    sorb, noA, noB = 100, 25, 25
    seeds = S.random_onvs(2, sorb, noA, noB, seed=44)
    comb = O.comb(seeds, sorb, noA, noB).reshape(-1, 16)
    rng = np.random.default_rng(45)
    keys = np.unique(np.concatenate([seeds, comb[rng.permutation(comb.shape[0])[:30000]]]), axis=0)
    psi = S.random_psi(keys.shape[0], seed=46)
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(sorb, seed=47, symmetric=False))
    lut = WavefunctionLUT(dev(keys), dev(psi), sorb, DEV, rank=0, world_size=1)
    x = dev(seeds)
    crow, col, val = csr(x, h1e, h2e, lut, sorb, noA + noB, noA, noB)
    check_structure(crow, col, keys.shape[0])
    assert np.diff(crow).min() > 10_000
    check_against_dense(crow, col, val, ops.get_hij_torch(x, lut.bra_key, h1e, h2e, sorb, noA + noB).cpu().numpy())
    check_eloc_identity(x, h1e, h2e, lut, sorb, noA + noB, noA, noB, crow, col, val)


# ---- 6. at scale: the benchmarked 10^6-sample Fe2S2 table ----------------------------------------------------------------
@gpu
@pytest.mark.parametrize("table", ["uniform", "zipf0.8"])
def test_headline_size_table(table):
    _need_gpu()
    import bench

    f = fe2s2()
    sorb, noA, noB, nele = int(f["sorb"]), int(f["noA"]), int(f["noB"]), int(f["nele"])
    keys = bench.make_table(table, 1_000_000)
    n = keys.shape[0]
    psi = S.random_psi(n, seed=1235)
    h1e, h2e = dev(np.ascontiguousarray(f["h1e"])), dev(np.ascontiguousarray(f["h2e"]))
    lut = WavefunctionLUT(dev(keys), dev(psi), sorb, DEV, rank=0, world_size=1)
    crow_d, col_d, val_d = ops.sample_space_hamiltonian(lut.bra_key, h1e, h2e, sorb, nele, noA, noB, lut.bra_key, lut.group_index)
    assert bool((crow_d[1:] >= crow_d[:-1]).all())
    # strictly ascending columns within every row (on the device: 3e7 entries)
    starts = torch.zeros(col_d.numel(), dtype=torch.bool, device=DEV)
    starts[crow_d[:-1][crow_d[:-1] < col_d.numel()]] = True
    assert bool(((col_d[1:] > col_d[:-1]) | starts[1:]).all())
    eloc, psi0 = ops.eloc_sample_space(lut.bra_key, h1e, h2e, sorb, nele, noA, noB, lut.bra_key, lut.wf_value, lut.group_index)
    Hs = torch.sparse_csr_tensor(crow_d, col_d, val_d, size=(n, n))
    Hpsi = torch.sparse.mm(Hs, lut.wf_value.view(-1, 1)).view(-1)
    want = eloc * psi0
    rel = ((Hpsi - want).abs() / want.abs()).max().item()
    assert rel < 1e-12
    w = psi0 * psi0 / (psi0 * psi0).sum()
    assert abs(float((w * Hpsi / psi0).sum() - (w * eloc).sum())) < 1e-10
    # a subsample of rows, the heaviest beta strings included, against dense get_hij_torch rows bitwise
    words = lut.bra_key.cpu().numpy().view(np.uint64).reshape(-1)
    rng = np.random.default_rng(7)
    pick = list(rng.choice(n, 250, replace=False))
    beta = words & np.uint64(0xAAAAAAAAAAAAAAAA)
    vals, counts = np.unique(beta, return_counts=True)
    for b in vals[np.argsort(counts)[-3:]]:
        pick += list(np.nonzero(beta == b)[0][[0, -1]])
    pick = np.array(sorted(set(int(i) for i in pick)))
    assert pick.size >= 250
    crow, col, val = crow_d.cpu().numpy(), col_d.cpu().numpy(), val_d.cpu().numpy()
    for chunk in np.array_split(pick, 8):
        H = ops.get_hij_torch(lut.bra_key[dev(chunk)], lut.bra_key, h1e, h2e, sorb, nele).cpu().numpy()
        sub_crow = np.concatenate([[0], np.cumsum(crow[chunk + 1] - crow[chunk])])
        sel = np.concatenate([np.arange(crow[i], crow[i + 1]) for i in chunk])
        check_against_dense(sub_crow, col[sel], val[sel], H)


# ---- 7. determinism, empty inputs, errors -----------------------------------------------------------------------------
@gpu
def test_determinism_sort_calls_and_empty_inputs():
    _need_gpu()
    f = fe2s2()
    sorb, nele, noA, noB = f["sorb"], f["nele"], f["noA"], f["noB"]
    lut = WavefunctionLUT(dev(f["ci"]), dev(S.random_psi(f["ci"].shape[0], seed=3)), sorb, DEV, rank=0, world_size=1)
    x = dev(f["ci"][:3000])
    h1e, h2e = dev(f["h1e"]), dev(f["h2e"])
    a = csr(x, h1e, h2e, lut, sorb, nele, noA, noB)
    b = csr(x, h1e, h2e, lut, sorb, nele, noA, noB)
    for u, v in zip(a, b):
        assert u.tobytes() == v.tobytes()
    nnz = int(a[0][-1])
    assert nnz > 3000
    _lib.set_tuning("sort_chunk", nnz // 7 + 1)  # the rows sorted in eight calls
    c = csr(x, h1e, h2e, lut, sorb, nele, noA, noB)
    for u, v in zip(a, c):
        assert u.tobytes() == v.tobytes()
    crow, col, val = ops.sample_space_hamiltonian(x[:0], h1e, h2e, sorb, nele, noA, noB, lut.bra_key, lut.group_index)
    assert crow.tolist() == [0] and col.numel() == 0 and val.numel() == 0
    crow, col, val = ops.sample_space_hamiltonian(x[:5], h1e, h2e, sorb, nele, noA, noB, lut.bra_key[:0])
    assert crow.tolist() == [0] * 6 and col.numel() == 0 and val.numel() == 0


@gpu
def test_bad_inputs_raise():
    _need_gpu()
    f = fe2s2()
    sorb, nele, noA, noB = f["sorb"], f["nele"], f["noA"], f["noB"]
    lut = WavefunctionLUT(dev(f["ci"]), dev(S.random_psi(f["ci"].shape[0], seed=3)), sorb, DEV, rank=0, world_size=1)
    x = dev(f["ci"][:10])
    h1e, h2e = dev(f["h1e"]), dev(f["h2e"])
    with pytest.raises(ValueError):
        ops.sample_space_hamiltonian(x, h1e.float(), h2e.float(), sorb, nele, noA, noB, lut.bra_key)
    with pytest.raises(ValueError):
        ops.sample_space_hamiltonian(torch.zeros((10, 16), dtype=torch.uint8, device=DEV), h1e, h2e, sorb, nele, noA, noB, lut.bra_key)
    other = WavefunctionLUT(dev(f["ci"][:100]), dev(np.ones(100)), sorb, DEV, rank=0, world_size=1)
    with pytest.raises(ValueError):
        ops.sample_space_hamiltonian(x, h1e, h2e, sorb, nele, noA, noB, lut.bra_key, other.group_index)
    # the C ABI refuses a scratch smaller than it asked for
    lib = _lib.load()
    nb = ctypes.c_int64()
    assert lib.pynqs_hamiltonian_scratch_bytes(_lib.i64(10), _lib.i64(0), sorb, noA, noB, ctypes.byref(nb)) == 0
    scratch = torch.empty(nb.value, dtype=torch.uint8, device=DEV)
    offsets = torch.empty(11, dtype=torch.int64, device=DEV)
    rc = lib.pynqs_hamiltonian_count(_lib.vp(x.data_ptr()), _lib.i64(10), sorb, noA, noB, _lib.vp(lut.bra_key.data_ptr()),
                                     _lib.i64(lut.bra_key.size(0)), _lib.vp(lut.group_index.workspace.data_ptr()), _lib.vp(scratch.data_ptr()),
                                     _lib.i64(nb.value - 1), _lib.vp(offsets.data_ptr()), _lib.vp(torch.cuda.current_stream().cuda_stream))
    assert rc == _lib.EWORKSPACE
    with pytest.raises(RuntimeError, match="scratch too small"):
        _lib.check(rc)
