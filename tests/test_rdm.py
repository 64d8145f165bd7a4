"""Reduced density matrices of sample-space states: energy.make_rdm1s / make_rdm12s over the pairs of the square CSR
sample-space Hamiltonian (pynqs_rdm_offdiag, C_extension.rdm_offdiag) plus the dense diagonal products.

The host oracle applies creation and annihilation operators literally to bit strings (the sign of get_hij_torch: an operator
on bit b counts the occupied bits below b).  It builds E_AB = a+_A a_B on a whole (n_alpha, n_beta) sector and takes
  dm1s[p, q] = c^H E_qp c,   dm2st[p, q, r, s] = (E_qp c)^H (E_rs c) - [s == t] [q == r] c^H E_ps c
(a+_p a+_r a_s a_q = E_pq E_rs - delta_qr E_ps), with c zero outside the table: the sample-space convention, in which only
the bra and the ket are restricted to the table.  On the host it is checked against oracle.hij (the energy), the closed form
of S^2 and the traces; on the GPU the device RDMs are checked against it element for element."""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from pynqs_b200 import C_extension as ops
from pynqs_b200 import _lib
from pynqs_b200 import synthetic as S
from pynqs_b200.energy import (local_energy_sample_space, make_rdm1s, make_rdm12s, sample_space_ground_state,
                               sample_space_hamiltonian, spin_square)
from pynqs_b200.lut import WavefunctionLUT

from test_spin_square import apply_op, closed_form, space, to_u8
from util import fe2s2

DEV = "cuda:0"
gpu = pytest.mark.gpu


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


# ---- the literal oracle ----------------------------------------------------------------------------------------------
def literal_rdm12(dets, c, sorb):
    """((dm1a, dm1b), (dm2aa, dm2ab, dm2bb)) of c (over dets, a whole sector as Python ints, zero outside the table),
    normalised by c^H c"""
    norb, D = sorb // 2, len(dets)
    idx = {d: k for k, d in enumerate(dets)}
    c = np.asarray(c)
    # Ec[s][a, b] = E_{a s, b s} c
    Ec = np.zeros((2, norb, norb, D), dtype=c.dtype)
    for s in range(2):
        for a in range(norb):
            for b in range(norb):
                for k, d in enumerate(dets):
                    for y, sg in apply_op(2 * a + s, True, apply_op(2 * b + s, False, {d: 1})).items():
                        Ec[s, a, b, idx[y]] += sg * c[k]
    norm = np.vdot(c, c).real
    dm1 = [np.einsum("k,qpk->pq", c.conj(), Ec[s]) / norm for s in range(2)]
    dm2 = []
    for s, t in ((0, 0), (0, 1), (1, 1)):
        U = Ec[s].transpose(1, 0, 2).reshape(norb * norb, D)  # row (p, q): E_qp c
        V = Ec[t].reshape(norb * norb, D)                      # row (r, s): E_rs c
        g = (U.conj() @ V.T).reshape(norb, norb, norb, norb) / norm
        if s == t:
            g -= np.einsum("qr,ps->pqrs", np.eye(norb), dm1[s].T)  # c^H E_ps c = dm1[s, p]
        dm2.append(g)
    return tuple(dm1), tuple(dm2)


def spatial_integrals(h1e, h2e, sorb):
    """h [norb, norb] and eri (pq|rs) [norb]^4 from the library's packed arrays: h[p, q] = h1e[2q sorb + 2p],
    (pq|rs) = <2p 2r+1||2q 2s+1> of the packed rule (an alpha-beta pair: no exchange term)"""
    norb = sorb // 2
    h = np.asarray(h1e).reshape(sorb, sorb)[0::2, 0::2].T.copy()
    p, q, r, s = np.meshgrid(*(np.arange(norb),) * 4, indexing="ij")
    i, j, k, l = 2 * p, 2 * r + 1, 2 * q, 2 * s + 1

    def pair(a, b):
        return np.where(a > b, a * (a - 1) // 2 + b, b * (b - 1) // 2 + a)

    ij, kl = pair(i, j), pair(k, l)
    sign = np.where(i > j, 1.0, -1.0) * np.where(k > l, 1.0, -1.0)
    hi, lo = np.maximum(ij, kl), np.minimum(ij, kl)
    return h, sign * np.asarray(h2e)[hi * (hi + 1) // 2 + lo]


def rdm_energy(dm1, dm2, h, eri):
    e = np.sum(h * (dm1[0] + dm1[1])) + 0.5 * np.sum(eri * dm2[0]) + np.sum(eri * dm2[1]) + 0.5 * np.sum(eri * dm2[2])
    return float(np.real(e))


def rdm_spin_square(dm1, dm2):
    """<S^2> = n_beta - sum_pq dm2ab[p, q, q, p] + Sz (Sz + 1)"""
    na, nb = np.trace(dm1[0]).real, np.trace(dm1[1]).real
    sz = (na - nb) / 2
    return float(nb - np.einsum("pqqp->", dm2[1]).real + sz * (sz + 1))


def check_traces(dm1, dm2, na, nb, atol):
    assert abs(np.trace(dm1[0]) - na) <= atol and abs(np.trace(dm1[1]) - nb) <= atol
    for g, want in zip(dm2, (na * (na - 1), na * nb, nb * (nb - 1))):
        assert abs(np.einsum("ppqq->", g) - want) <= atol * max(1, want)


def fe2s2_prefix():
    """the first 12 spin orbitals of the Fe2S2 integrals: the packed pairs below orbital 12 are a prefix of h2e"""
    f = fe2s2()
    return f["h1e"].reshape(40, 40)[:12, :12].copy().reshape(-1), f["h2e"][:2211].copy()


def ints_of(u8):
    w = u8.view(np.uint64).reshape(u8.shape[0], -1)
    return [sum(int(v) << (64 * k) for k, v in enumerate(row)) for row in w]


def random_c(n, seed, cplx):
    rng = np.random.default_rng(seed)
    c = rng.standard_normal(n) + (1j * rng.standard_normal(n) if cplx else 0)
    return c / np.linalg.norm(c)


# ---- host checks -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("half", [False, True])
def test_literal_oracle_identities(cplx, half):
    """energy, <S^2> and traces of the literal RDMs on the 12-orbital Fe2S2 prefix, 3a3b (400 determinants), against
    oracle.hij and the closed form of S^2 over the same table"""
    sorb, na, nb = 12, 3, 3
    h1e, h2e = fe2s2_prefix()
    dets = sorted(space(sorb, na, nb))
    assert len(dets) == 400
    rng = np.random.default_rng(11)
    table = sorted(dets[k] for k in rng.permutation(400)[:200]) if half else dets
    key = to_u8(table, sorb)
    ct = random_c(len(table), 12 + cplx, cplx)
    c = np.zeros(len(dets), dtype=ct.dtype)
    c[[dets.index(d) for d in table]] = ct
    dm1, dm2 = literal_rdm12(dets, c, sorb)
    H = O.hij(key, key, h1e, h2e, sorb, na + nb)
    h, eri = spatial_integrals(h1e, h2e, sorb)
    e = float(np.real(ct.conj() @ H @ ct))
    assert abs(rdm_energy(dm1, dm2, h, eri) - e) <= 1e-12 * abs(e)
    s2 = float(np.real(ct.conj() @ (closed_form(key, key, sorb) @ ct)))
    assert abs(rdm_spin_square(dm1, dm2) - s2) <= 1e-12
    check_traces(dm1, dm2, na, nb, 1e-12)
    np.testing.assert_allclose(dm1[0], dm1[0].conj().T, rtol=0, atol=1e-15)


def test_rdm_offdiag_bad_arguments_on_the_cpu():
    lib = _lib.load()
    p = _lib.vp(256)  # never dereferenced: the checks come first
    null = _lib.vp(None)

    def call(crow=p, col=p, key=p, N=10, nnz=40, sorb=40, c=p, cplx=0, sc=p, nbytes=1 << 30, dm1=p, dm2=p):
        return lib.pynqs_rdm_offdiag(crow, col, key, _lib.i64(N), _lib.i64(nnz), int(sorb), c, int(cplx), sc, _lib.i64(nbytes), dm1, dm2, null)

    for bad in (dict(N=-1), dict(N=1 << 31), dict(nnz=-1), dict(nnz=1 << 31), dict(sorb=0), dict(sorb=41), dict(sorb=194),
                dict(cplx=2), dict(dm1=null), dict(crow=null), dict(key=null), dict(c=null), dict(col=null), dict(sc=null)):
        assert call(**bad) == _lib.EVALUE, bad
    assert b"rdm_offdiag" in lib.pynqs_last_error()
    nb = _lib.ctypes.c_int64()
    assert lib.pynqs_rdm_scratch_bytes(_lib.i64(10), _lib.i64(-1), 40, _lib.ctypes.byref(nb)) == _lib.EVALUE
    assert lib.pynqs_rdm_scratch_bytes(_lib.i64(10), _lib.i64(40), 39, _lib.ctypes.byref(nb)) == _lib.EVALUE
    assert lib.pynqs_rdm_scratch_bytes(_lib.i64(10), _lib.i64(40), 40, null) == _lib.EVALUE
    assert lib.pynqs_rdm_scratch_bytes(_lib.i64(10), _lib.i64(1000), 40, _lib.ctypes.byref(nb)) == 0
    assert 30 * 1000 + (4 << 20) <= nb.value <= 30 * 1000 + (4 << 20) + 8 * 256
    u8 = torch.zeros(4, 8, dtype=torch.uint8)
    crow = torch.zeros(5, dtype=torch.int64)
    with pytest.raises(NotImplementedError):
        ops.rdm_offdiag(crow, crow[:0], u8, torch.zeros(4, dtype=torch.float64), 40)


# ---- the device RDMs -------------------------------------------------------------------------------------------------
def table(keys, sorb, seed=1, cplx=False):
    return WavefunctionLUT(dev(keys), dev(S.random_psi(keys.shape[0], seed=seed, complex_=cplx)), sorb, DEV, rank=0, world_size=1)


def square_h(lut, sorb, na, nb, seed=21):
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(sorb, seed=seed, symmetric=True))
    return sample_space_hamiltonian(lut.bra_key, h1e, h2e, lut, sorb, na + nb, na, nb)


def device_rdm12(lut, c, sorb, H):
    (a, b), (aa, ab, bb) = make_rdm12s(lut, c, sorb, H)
    return tuple(t.cpu().numpy() for t in (a, b)), tuple(t.cpu().numpy() for t in (aa, ab, bb))


def assert_rdms_close(got, want, atol):
    for g, w in zip(got[0] + got[1], want[0] + want[1]):
        assert g.shape == w.shape
        np.testing.assert_allclose(g, w, rtol=0, atol=atol)


@gpu
@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("sorb,na,nb,half", [(10, 3, 2, False), (12, 3, 3, False), (14, 4, 2, False), (12, 3, 3, True)])
def test_matches_literal_oracle(sorb, na, nb, half, cplx):
    _need_gpu()
    dets = sorted(space(sorb, na, nb))
    if half:
        rng = np.random.default_rng(3)
        dets_t = sorted(dets[k] for k in rng.permutation(len(dets))[: len(dets) // 2])
    else:
        dets_t = dets
    lut = table(to_u8(dets_t, sorb), sorb)
    order = ints_of(lut.bra_key.cpu().numpy())
    ct = random_c(len(order), sorb + half, cplx)
    c = np.zeros(len(dets), dtype=ct.dtype)
    c[[dets.index(d) for d in order]] = ct
    want = literal_rdm12(dets, c, sorb)
    H = square_h(lut, sorb, na, nb)
    got = device_rdm12(lut, dev(ct), sorb, H)
    assert got[0][0].dtype == ct.dtype
    assert_rdms_close(got, want, 1e-12)
    d1 = make_rdm1s(lut, dev(ct), sorb, H)
    for g, w in zip(d1, got[0]):
        assert g.cpu().numpy().tobytes() == w.tobytes()


@gpu
@pytest.mark.parametrize("sorb", [100, 140])
def test_multi_word_onvs(sorb):
    """Two- and three-word ONVs: 7 orbitals placed across the words (an increasing map, so the signs are those of the
    7-orbital space), a table of two determinants and all their singles and doubles, against the oracle on the 7-orbital
    sector scattered to the mapped orbitals"""
    _need_gpu()
    small, na, nb = 14, 3, 2
    pos = [1, 20, 31, 32, 40, 55, 69][: small // 2] if sorb == 140 else [0, 15, 31, 32, 33, 47, 49]
    dets = sorted(space(small, na, nb))
    base = [dets[5], dets[-9]]
    near = sorted({d for d in dets for b in base if bin(d ^ b).count("1") <= 4})
    assert len(near) < len(dets)

    def widen(d):
        return sum(1 << (2 * pos[k] + s) for k in range(small // 2) for s in range(2) if (d >> (2 * k + s)) & 1)

    wide = {widen(d): d for d in near}
    lut = table(to_u8(sorted(wide), sorb), sorb)
    order = [wide[d] for d in ints_of(lut.bra_key.cpu().numpy())]
    for cplx in (False, True):
        ct = random_c(len(order), sorb + cplx, cplx)
        c = np.zeros(len(dets), dtype=ct.dtype)
        c[[dets.index(d) for d in order]] = ct
        w1, w2 = literal_rdm12(dets, c, small)
        n = sorb // 2
        ix = np.ix_(pos, pos)
        want1 = tuple(np.zeros((n, n), ct.dtype) for _ in range(2))
        want2 = tuple(np.zeros((n,) * 4, ct.dtype) for _ in range(3))
        for a, b in zip(want1, w1):
            a[ix] = b
        for a, b in zip(want2, w2):
            a[np.ix_(pos, pos, pos, pos)] = b
        got = device_rdm12(lut, dev(ct), sorb, square_h(lut, sorb, na, nb))
        assert_rdms_close(got, (want1, want2), 1e-12)


@gpu
def test_fe2s2_ci_ground_state():
    _need_gpu()
    f = fe2s2()
    sorb, nele, na, nb = f["sorb"], f["nele"], f["noA"], f["noB"]
    lut = table(f["ci"], sorb, seed=3)
    h1e, h2e = dev(f["h1e"]), dev(f["h2e"])
    H = sample_space_hamiltonian(lut.bra_key, h1e, h2e, lut, sorb, nele, na, nb)
    e, C, info = sample_space_ground_state(lut, h1e, h2e, sorb, nele, na, nb, H=H)
    assert info["converged"]
    c = C[:, 0].contiguous()
    dm1, dm2 = device_rdm12(lut, c, sorb, H)
    h, eri = spatial_integrals(f["h1e"], f["h2e"], sorb)
    cHc = float(c @ ops.csr_matmul(H.crow_indices(), H.col_indices(), H.values(), c, c.numel())) / float(c @ c)
    assert abs(rdm_energy(dm1, dm2, h, eri) - cHc) <= 1e-12 * abs(cHc)
    s2 = float(spin_square(lut, c, sorb)[0])
    assert abs(s2 - 6.0) < 1e-6  # the quintet
    assert abs(rdm_spin_square(dm1, dm2) - s2) <= 1e-10
    check_traces(dm1, dm2, na, nb, 1e-10)
    for d in dm1:
        w = np.linalg.eigvalsh(d)
        assert w.min() >= -1e-12 and w.max() <= 1 + 1e-12
    occ = np.linalg.eigvalsh(dm1[0] + dm1[1])
    assert occ.min() >= -1e-12 and occ.max() <= 2 + 1e-12 and abs(occ.sum() - nele) <= 1e-10


@gpu
@pytest.mark.parametrize("cplx", [False, True])
def test_uniform_table_of_10_6_samples(cplx):
    _need_gpu()
    import bench

    h1e_np, h2e_np, _ = bench.load_integrals()
    sorb, nele, na, nb = bench.SORB, bench.NELE, bench.NOA, bench.NOB
    keys = bench.make_table("uniform", 1_000_000)
    lut = table(keys, sorb, seed=4, cplx=cplx)
    h1e, h2e = dev(h1e_np), dev(h2e_np)
    H = sample_space_hamiltonian(lut.bra_key, h1e, h2e, lut, sorb, nele, na, nb)
    psi = lut.wf_value
    dm1, dm2 = device_rdm12(lut, psi, sorb, H)
    eloc, _, psi_x = local_energy_sample_space(lut.bra_key, h1e, h2e, lut, sorb, nele, na, nb, dtype=psi.dtype)
    w = psi_x.abs() ** 2
    e = float((w * eloc.real).sum() / w.sum()) if cplx else float((w * eloc).sum() / w.sum())
    h, eri = spatial_integrals(h1e_np, h2e_np, sorb)
    assert abs(rdm_energy(dm1, dm2, h, eri) - e) <= 1e-11 * abs(e)
    assert abs(rdm_spin_square(dm1, dm2) - float(spin_square(lut, psi, sorb)[0])) <= 1e-10
    check_traces(dm1, dm2, na, nb, 1e-10)
    again = device_rdm12(lut, psi, sorb, H)
    for a, b in zip(dm1 + dm2, again[0] + again[1]):
        assert a.tobytes() == b.tobytes()
    for a, b in zip(make_rdm1s(lut, psi, sorb, H), dm1):
        assert a.cpu().numpy().tobytes() == b.tobytes()


@gpu
def test_one_row_table():
    """dm1 is the occupations, dm2 the occupation products with their exchange signs"""
    _need_gpu()
    sorb = 12
    d = space(sorb, 3, 2)[7]
    lut = table(to_u8([d], sorb), sorb)
    H = square_h(lut, sorb, 3, 2)
    c = torch.tensor([-0.5], dtype=torch.float64, device=DEV)
    (a, b), (aa, ab, bb) = (tuple(t.cpu().numpy() for t in x) for x in make_rdm12s(lut, c, sorb, H))
    n = np.array([[(d >> (2 * p + s)) & 1 for p in range(sorb // 2)] for s in range(2)], dtype=np.float64)
    np.testing.assert_array_equal(a, np.diag(n[0]))
    np.testing.assert_array_equal(b, np.diag(n[1]))
    for g, (s, t) in zip((aa, ab, bb), ((0, 0), (0, 1), (1, 1))):
        want = np.zeros((sorb // 2,) * 4)
        for p in range(sorb // 2):
            for r in range(sorb // 2):
                if s != t or p != r:
                    want[p, p, r, r] = n[s, p] * n[t, r]
                    if s == t:
                        want[p, r, r, p] = -n[s, p] * n[t, r]
        np.testing.assert_array_equal(g, want)


@gpu
def test_value_errors():
    _need_gpu()
    sorb = 12
    lut = table(to_u8(space(sorb, 3, 3), sorb), sorb)
    H = square_h(lut, sorb, 3, 3)
    c = lut.wf_value
    with pytest.raises(ValueError):
        make_rdm12s(lut, c, sorb, H.to_dense())  # not CSR
    Hr = sample_space_hamiltonian(lut.bra_key[:10], *(dev(a) for a in S.random_packed_integrals(sorb, seed=21, symmetric=True)), lut,
                                  sorb, 6, 3, 3)
    with pytest.raises(ValueError):
        make_rdm12s(lut, c, sorb, Hr)  # (10, N)
    with pytest.raises(ValueError):
        make_rdm12s(lut, c[:399], sorb, H)
    with pytest.raises(ValueError):
        make_rdm1s(lut, c.float(), sorb, H)
    with pytest.raises(ValueError):
        make_rdm12s(lut, torch.zeros_like(c), sorb, H)
    keys = lut.bra_key.cpu().numpy()
    dup = table(np.concatenate([keys[:50], keys[40:60]]), sorb)
    assert (dup.bra_key[1:] == dup.bra_key[:-1]).all(1).any()
    Hd = square_h(dup, sorb, 3, 3)
    with pytest.raises(ValueError, match="duplicate"):
        make_rdm1s(dup, dup.wf_value, sorb, Hd)
