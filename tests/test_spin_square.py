"""Total spin over the sample space: S^2 X over the sorted table (pynqs_spin_square_apply / C_extension.spin_square_matmul),
the local spin S^2_loc and <S^2> (energy.local_spin_square / spin_square), and spin-targeted roots
(energy.sample_space_ground_state with spin_shift / ss).

The host oracle applies S+ and S- literally to bit strings (creation / annihilation operators with the sign of
get_hij_torch: an operator on bit b counts the occupied bits below b).  It checks, on full spaces, the vectorised closed form
that the GPU tests compare with on large tables: <x|S^2|x> = |B| + Sz (Sz + 1) and +1 for each spin exchange of an
alpha-only orbital p and a beta-only orbital q (A / B: the alpha-only / beta-only orbitals of x)."""
import itertools
from math import comb

import numpy as np
import pytest
import scipy.sparse
import scipy.sparse.linalg
import torch

from oracle import oracle as O
from pynqs_b200 import C_extension as ops
from pynqs_b200 import _lib
from pynqs_b200 import synthetic as S
from pynqs_b200.energy import local_spin_square, sample_space_ground_state, sample_space_hamiltonian, spin_square
from pynqs_b200.lut import WavefunctionLUT

from util import fe2s2

DEV = "cuda:0"
gpu = pytest.mark.gpu

# lowest three eigenvalues of H over the Fe2S2 CI space (tests/test_sample_space_ground_state.py) and their spins S, from
# scipy.sparse.linalg.eigsh on the host matrix and <S^2> = S (S + 1) with the host closed form below.  The space has at most
# four open shells, so S <= 2 in it.
FE2S2_CI_LOWEST = [-114.3785426621286, -114.35772955847762, -114.34255940058875]
FE2S2_CI_SPINS = [2, 1, 2]


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def space(sorb, noA, noB):
    """every determinant with noA alpha and noB beta electrons in sorb spin orbitals, as Python ints"""
    half = sorb // 2
    a = [sum(1 << (2 * k) for k in c) for c in itertools.combinations(range(half), noA)]
    b = [sum(1 << (2 * k + 1) for k in c) for c in itertools.combinations(range(half), noB)]
    return [x | y for x in a for y in b]


def to_u8(ints, sorb):
    L = (sorb - 1) // 64 + 1
    return np.array([[(v >> (64 * w)) & (2**64 - 1) for w in range(L)] for v in ints], dtype=np.uint64).view(np.uint8).reshape(-1, 8 * L)


# ---- the literal operator ------------------------------------------------------------------------------------------
def apply_op(bit, create, state):
    """a+_bit (create) or a_bit on the linear combination state {determinant: coefficient}"""
    out = {}
    for x, c in state.items():
        if bool((x >> bit) & 1) == create:
            continue
        sign = -1 if bin(x & ((1 << bit) - 1)).count("1") & 1 else 1
        y = x ^ (1 << bit)
        out[y] = out.get(y, 0) + sign * c
    return out


def add(u, v, scale=1):
    out = dict(u)
    for x, c in v.items():
        out[x] = out.get(x, 0) + scale * c
    return out


def s_plus(norb, state):  # sum_p a+_{p alpha} a_{p beta}
    out = {}
    for p in range(norb):
        out = add(out, apply_op(2 * p, True, apply_op(2 * p + 1, False, state)))
    return out


def s_minus(norb, state):  # sum_p a+_{p beta} a_{p alpha}
    out = {}
    for p in range(norb):
        out = add(out, apply_op(2 * p + 1, True, apply_op(2 * p, False, state)))
    return out


def s_z(norb, state):  # (n_alpha - n_beta) / 2, from the number operators
    out = {}
    for p in range(norb):
        out = add(out, apply_op(2 * p, True, apply_op(2 * p, False, state)), 0.5)
        out = add(out, apply_op(2 * p + 1, True, apply_op(2 * p + 1, False, state)), -0.5)
    return out


def literal_s2(norb, x):
    """S^2 |x> = S- S+ |x> + Sz (Sz + 1) |x>"""
    v = {x: 1}
    sz = s_z(norb, v)
    out = add(s_minus(norb, s_plus(norb, v)), s_z(norb, sz))
    return {y: c for y, c in add(out, sz).items() if c != 0}


def literal_matrix(dets, sorb):
    idx = {d: i for i, d in enumerate(dets)}
    M = np.zeros((len(dets), len(dets)))
    for j, d in enumerate(dets):
        for y, c in literal_s2(sorb // 2, d).items():
            M[idx[y], j] += c
    return M


# ---- the vectorised closed form --------------------------------------------------------------------------------------
def classic_search(keys, q):
    """row of every query in the sorted table (the reference's binary search, so with duplicate keys the row it lands
    on), -1 if absent; keys uint64 [N, L], q uint64 [m, L] (word L - 1 most significant)"""
    N, m = keys.shape[0], q.shape[0]
    lo, hi = np.zeros(m, np.int64), np.full(m, N - 1, np.int64)
    res = np.full(m, -1, np.int64)
    active = np.ones(m, bool)
    while True:
        active &= lo <= hi
        if not active.any():
            return res
        mid = lo + (hi - lo) // 2
        e = keys[np.where(active, mid, 0)]
        c = np.zeros(m, np.int64)
        for w in range(q.shape[1]):  # the most significant differing word decides
            c = np.where(e[:, w] < q[:, w], -1, np.where(e[:, w] > q[:, w], 1, c))
        found = active & (c == 0)
        res[found] = mid[found]
        active &= ~found
        lo = np.where(active & (c < 0), mid + 1, lo)
        hi = np.where(active & (c > 0), mid - 1, hi)


def spin_exchanges(bra, sorb):
    """(row of the bra, partner uint64 [m, L]) of every spin exchange of every bra, rows ascending, (p, q) ascending inside
    a row; and the diagonal <x|S^2|x> of every bra"""
    n, L = bra.shape[0], bra.shape[1] // 8
    bits = np.unpackbits(bra, axis=1, bitorder="little")[:, :sorb].astype(bool)
    oa, ob = bits[:, 0::2], bits[:, 1::2]
    A, B = oa & ~ob, ob & ~oa
    sz2 = oa.sum(1).astype(np.int64) - ob.sum(1)
    diag = B.sum(1) + sz2 * (sz2 + 2) / 4.0
    rows, p, q = np.nonzero(A[:, :, None] & B[:, None, :])
    norb = sorb // 2
    flip = np.zeros((norb, L), np.uint64)
    flip[np.arange(norb), (2 * np.arange(norb)) // 64] = np.uint64(3) << ((2 * np.arange(norb)) % 64).astype(np.uint64)
    words = bra.view(np.uint64).reshape(n, L)
    return rows, words[rows] ^ flip[p] ^ flip[q], diag


def closed_form(bra, key, sorb):
    """S^2 over the table as scipy CSR [n, N], with the kernel's conventions: the diagonal where bra_i is in the table,
    +1 where a spin exchange is; the row the classic search lands on for duplicate keys"""
    n, N, L = bra.shape[0], key.shape[0], bra.shape[1] // 8
    kw = key.view(np.uint64).reshape(N, L)
    rows, partners, diag = spin_exchanges(bra, sorb)
    self_col = classic_search(kw, bra.view(np.uint64).reshape(n, L))
    cols = classic_search(kw, partners)
    r = np.concatenate([np.nonzero(self_col >= 0)[0], rows[cols >= 0]])
    c = np.concatenate([self_col[self_col >= 0], cols[cols >= 0]])
    v = np.concatenate([diag[self_col >= 0], np.ones(int((cols >= 0).sum()))])
    return scipy.sparse.csr_matrix((v, (r, c)), shape=(n, N))


def multiplicities(norb, noA, noB):
    """{S(S + 1): number of spin-S states} in the sector: D(M) - D(M + 1) with D(M) the number of determinants of Sz = M"""
    n, sz = noA + noB, (noA - noB) / 2

    def D(M):
        na = round(n / 2 + M)
        nb = n - na
        return comb(norb, na) * comb(norb, nb) if 0 <= na <= norb and 0 <= nb <= norb else 0

    out, s = {}, abs(sz)
    while D(s) > 0:
        if D(s) - D(s + 1):
            out[s * (s + 1)] = D(s) - D(s + 1)
        s += 1
    return out


# ---- host checks ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sorb,noA,noB", [(10, 3, 2), (12, 3, 3), (14, 4, 2)])
def test_literal_operator_matches_the_closed_form(sorb, noA, noB):
    dets = sorted(space(sorb, noA, noB))
    M = literal_matrix(dets, sorb)
    u8 = to_u8(dets, sorb)
    C = closed_form(u8, u8, sorb).toarray()
    assert np.array_equal(M, C)
    off = M - np.diag(np.diag(M))
    assert set(np.unique(off)) <= {0.0, 1.0}  # every spin exchange has the element +1
    if (sorb, noA, noB) == (12, 3, 3):
        assert len(dets) == 400


@pytest.mark.parametrize("sorb,noA,noB", [(10, 3, 2), (12, 3, 3), (14, 4, 2)])
def test_spectrum_is_s_s_plus_1_with_multiplicities(sorb, noA, noB):
    M = literal_matrix(sorted(space(sorb, noA, noB)), sorb)
    w = np.linalg.eigvalsh(M)
    vals, counts = np.unique(np.round(w, 8), return_counts=True)
    assert np.abs(w - np.round(w * 4) / 4).max() < 1e-10
    assert dict(zip(vals.tolist(), counts.tolist())) == multiplicities(sorb // 2, noA, noB)


def test_closed_form_with_duplicates_and_rows_outside_the_table():
    """the vectorised form against the literal operator where the table is a part of the space: entries only where the
    column is in the table, duplicate keys resolved to the classic search's row"""
    dets = sorted(space(10, 3, 2))
    rng = np.random.default_rng(5)
    table = sorted([dets[i] for i in rng.permutation(len(dets))[:60]] + [dets[i] for i in rng.permutation(len(dets))[:10]])
    key = to_u8(table, 10)
    M = closed_form(to_u8(dets, 10), key, 10).toarray()
    row = classic_search(key.view(np.uint64).reshape(-1, 1), np.array(dets, np.uint64).reshape(-1, 1))
    for i, d in enumerate(dets):
        want = np.zeros(len(table))
        for y, c in literal_s2(5, d).items():
            j = row[dets.index(y)]
            if j >= 0:
                want[j] += c
        assert np.array_equal(M[i], want), i


def test_spin_square_apply_bad_arguments_on_the_cpu():
    lib = _lib.load()
    p = _lib.vp(256)  # never dereferenced: the checks come first

    def call(bra=p, n=10, sorb=40, key=p, N=10, ws=p, X=p, ldx=2, k=2, Y=p, ldy=2):
        return lib.pynqs_spin_square_apply(bra, _lib.i64(n), int(sorb), key, _lib.i64(N), ws, X, _lib.i64(ldx), int(k), Y, _lib.i64(ldy),
                                           _lib.vp(None))

    null = _lib.vp(None)
    for bad in (dict(n=-1), dict(N=-1), dict(N=1 << 31), dict(k=0), dict(k=9, ldx=9, ldy=9), dict(ldx=1), dict(ldy=1), dict(sorb=0),
                dict(sorb=41), dict(sorb=194), dict(bra=null), dict(Y=null), dict(key=null), dict(ws=null), dict(X=null)):
        assert call(**bad) == _lib.EVALUE, bad
    assert b"spin_square_apply" in lib.pynqs_last_error()
    assert call(n=0, bra=null, key=null, ws=null, X=null, Y=null) == 0  # no rows: nothing to do, nothing launched
    u8 = torch.zeros(4, 8, dtype=torch.uint8)
    with pytest.raises(NotImplementedError):
        ops.spin_square_matmul(u8, 40, u8, torch.zeros(4, dtype=torch.float64))


# ---- the product on the GPU ------------------------------------------------------------------------------------------
def check_product(bra, lut, sorb, seed, M=None):
    """spin_square_matmul(bra, ...) against the host closed form for k = 1, 3, 8, 11, a 1-D vector and a complex block,
    each twice with identical bits.  Returns the host matrix."""
    if M is None:
        M = closed_form(bra, lut.bra_key.cpu().numpy(), sorb)
    absM = abs(M)
    N = lut.bra_key.size(0)
    rng = np.random.default_rng(seed)
    bra_d = dev(bra)

    def agree(X):
        Y = ops.spin_square_matmul(bra_d, sorb, lut.bra_key, dev(X), lut.group_index)
        want = M @ X
        assert Y.shape == want.shape and Y.dtype == torch.from_numpy(want).dtype
        Yh = Y.cpu().numpy()
        assert (np.abs(Yh - want) <= 1e-14 * (absM @ np.abs(X)) + 1e-300).all()
        assert Yh.tobytes() == ops.spin_square_matmul(bra_d, sorb, lut.bra_key, dev(X), lut.group_index).cpu().numpy().tobytes()

    for k in (1, 3, 8, 11):
        agree(rng.standard_normal((N, k)))
    agree(rng.standard_normal(N))
    agree(rng.standard_normal((N, 3)) + 1j * rng.standard_normal((N, 3)))
    return M


def table(keys, sorb, seed=1, cplx=False):
    return WavefunctionLUT(dev(keys), dev(S.random_psi(keys.shape[0], seed=seed, complex_=cplx)), sorb, DEV, rank=0, world_size=1)


def check_every_partner_found(lut, sorb, M):
    """S^2 applied to ones on the square table counts the diagonal and the partners of every row: all of them are found"""
    key = lut.bra_key.cpu().numpy()
    rows, _, diag = spin_exchanges(key, sorb)
    ones = ops.spin_square_matmul(lut.bra_key, sorb, lut.bra_key, torch.ones(key.shape[0], dtype=torch.float64, device=DEV))
    np.testing.assert_array_equal(ones.cpu().numpy(), diag + np.bincount(rows, minlength=key.shape[0]))
    np.testing.assert_array_equal(M @ np.ones(key.shape[0]), diag + np.bincount(rows, minlength=key.shape[0]))
    return rows


@gpu
def test_full_space_every_partner_found():
    _need_gpu()
    lut = table(to_u8(space(12, 3, 3), 12), 12)
    M = check_product(lut.bra_key.cpu().numpy(), lut, 12, seed=1)
    check_every_partner_found(lut, 12, M)


@gpu
def test_fe2s2_ci_space_is_spin_complete():
    _need_gpu()
    f = fe2s2()
    lut = table(f["ci"], f["sorb"])
    key = lut.bra_key.cpu().numpy()
    rows, partners, _ = spin_exchanges(key, f["sorb"])
    assert rows.size == 61200 and np.bincount(rows).max() == 4
    assert (classic_search(key.view(np.uint64).reshape(-1, 1), partners) >= 0).all()  # every partner is in the space
    M = check_product(key, lut, f["sorb"], seed=2)
    check_every_partner_found(lut, f["sorb"], M)


@gpu
def test_uniform_table_of_10_5_samples():
    _need_gpu()
    import bench

    keys = bench.make_table("uniform", 100_000)
    lut = table(keys, bench.SORB, seed=3)
    M = check_product(lut.bra_key.cpu().numpy(), lut, bench.SORB, seed=3)
    rows, _, _ = spin_exchanges(lut.bra_key.cpu().numpy(), bench.SORB)
    assert np.bincount(rows).max() <= 25 and M.nnz < 100_000 + rows.size  # most partners are not in the table


@gpu
def test_rectangular_mixed_sectors_half_outside_the_table():
    """bras half inside, half outside a table that mixes (noA, noB) sectors of integer and half-integer Sz"""
    _need_gpu()
    dets = space(12, 3, 3) + space(12, 4, 2) + space(12, 2, 3) + space(12, 5, 1)
    rng = np.random.default_rng(7)
    perm = rng.permutation(len(dets))
    keys = to_u8([dets[i] for i in perm[: len(dets) // 2]], 12)
    bra = to_u8([dets[i] for i in perm[len(dets) // 4 : 3 * len(dets) // 4]], 12)
    lut = table(keys, 12, seed=4)
    M = check_product(bra, lut, 12, seed=4)
    inside = classic_search(lut.bra_key.cpu().numpy().view(np.uint64).reshape(-1, 1), bra.view(np.uint64).reshape(-1, 1)) >= 0
    assert inside[: len(dets) // 4].all() and not inside[len(dets) // 4 :].any()
    assert M[np.nonzero(~inside)[0]].nnz > 0  # bras outside the table still reach partners inside it


@gpu
def test_table_with_duplicate_keys():
    _need_gpu()
    dets = space(10, 3, 2)
    rng = np.random.default_rng(8)
    picks = [dets[i] for i in rng.permutation(len(dets))[:60]] + [dets[i] for i in rng.permutation(len(dets))[:15]]
    keys = to_u8(picks, 10)
    lut = table(keys, 10, seed=5)
    k = lut.bra_key.cpu().numpy().view(np.uint64).reshape(-1)
    assert (k[1:] == k[:-1]).any()
    check_product(to_u8(dets, 10), lut, 10, seed=5)


@gpu
@pytest.mark.parametrize("sorb", [100, 140])
def test_multi_word_onvs(sorb):
    """Two- and three-word ONVs (6 alpha, 4 beta electrons): a small random table into which the spin exchanges of some
    samples have been inserted, partners across word boundaries included"""
    _need_gpu()
    samples = S.random_onvs(400, sorb, 6, 4, seed=sorb)
    rows, partners, _ = spin_exchanges(samples[:60], sorb)
    L = samples.shape[1] // 8
    pick = np.random.default_rng(sorb + 1).random(rows.size) < 0.7
    keys = np.unique(np.concatenate([samples[:300], partners[pick].view(np.uint8).reshape(-1, 8 * L)]), axis=0)
    lut = table(keys, sorb, seed=6)
    M = check_product(samples, lut, sorb, seed=6)
    assert M[:60].nnz >= 60 + pick.sum()
    changed = np.count_nonzero(partners != samples[:60].view(np.uint64).reshape(60, L)[rows], axis=1)
    assert (changed == 2).any()  # some spin exchanges span two words


@gpu
def test_spin_square_matmul_empty_and_bad_inputs():
    _need_gpu()
    keys = to_u8(space(12, 3, 3), 12)
    lut = table(keys, 12)
    bra = lut.bra_key
    l0 = _lib.launch_count()
    y = ops.spin_square_matmul(bra[:0], 12, bra, torch.ones(400, 2, dtype=torch.float64, device=DEV))
    assert y.shape == (0, 2)
    empty = torch.zeros(0, 8, dtype=torch.uint8, device=DEV)
    y = ops.spin_square_matmul(bra, 12, empty, torch.zeros(0, dtype=torch.complex128, device=DEV))
    assert y.shape == (400,) and y.dtype == torch.complex128 and not y.any()
    assert _lib.launch_count() == l0  # nothing to do, nothing launched
    x = torch.ones(400, dtype=torch.float64, device=DEV)
    with pytest.raises(ValueError):
        ops.spin_square_matmul(bra, 12, bra, x.float())
    with pytest.raises(ValueError):
        ops.spin_square_matmul(bra, 12, bra, x[:399])
    with pytest.raises(ValueError):
        ops.spin_square_matmul(bra, 100, bra, x)  # width of a one-word ONV, sorb of two words
    other = table(keys[::-1].copy(), 12)
    with pytest.raises(ValueError):
        ops.spin_square_matmul(bra, 12, bra, x, other.group_index)


# ---- local spin and <S^2> ----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("cplx", [False, True])
def test_local_spin_square(cplx):
    _need_gpu()
    f = fe2s2()
    sorb = f["sorb"]
    lut = table(f["ci"], sorb, seed=9, cplx=cplx)
    outside = S.random_onvs(50, sorb, f["noA"], f["noB"], seed=10)
    x = torch.cat([lut.bra_key[:500], dev(outside)])
    inside = (classic_search(lut.bra_key.cpu().numpy().view(np.uint64).reshape(-1, 1), outside.view(np.uint64).reshape(-1, 1)) >= 0)
    s2loc, psi_x = local_spin_square(x, lut, sorb)
    assert s2loc.dtype == lut.wf_value.dtype and psi_x.dtype == lut.wf_value.dtype
    s2psi = ops.spin_square_matmul(x, sorb, lut.bra_key, lut.wf_value).cpu().numpy()
    s, p = s2loc.cpu().numpy(), psi_x.cpu().numpy()
    have = np.concatenate([np.ones(500, bool), inside])
    np.testing.assert_array_equal(p[:500], lut.wf_value[:500].cpu().numpy())
    assert (np.abs(s[have] * p[have] - s2psi[have]) <= 1e-14 * np.abs(s2psi[have]) + 1e-300).all()
    assert (~have).any() and (p[~have] == 0).all() and np.isnan(s[~have]).all()
    # the |psi|^2-weighted mean over the table is <S^2> of psi
    s2loc, psi_x = local_spin_square(lut.bra_key, lut, sorb)
    w = psi_x.abs() ** 2
    mean = float(((w * s2loc).sum() / w.sum()).real)
    want = spin_square(lut, lut.wf_value, sorb)
    assert want.shape == (1,) and abs(mean - float(want[0])) <= 1e-12 * abs(float(want[0]))


# ---- spin of the roots ------------------------------------------------------------------------------------------------
def nearest_s(v):
    s = (np.sqrt(1 + 4 * np.asarray(v)) - 1) / 2  # s (s + 1) = v
    return np.round(s)


@gpu
def test_full_space_roots_are_spin_eigenstates():
    _need_gpu()
    keys = to_u8(space(12, 3, 3), 12)
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(12, seed=21, symmetric=True))
    lut = table(keys, 12)
    e, C, info = sample_space_ground_state(lut, h1e, h2e, 12, 6, 3, 3, nroots=6)
    assert info["converged"]
    s2 = spin_square(lut, C, 12).cpu().numpy()
    s = nearest_s(s2)
    assert np.abs(s2 - s * (s + 1)).max() <= 1e-9


@gpu
def test_fe2s2_ci_lowest_three_spins():
    _need_gpu()
    f = fe2s2()
    sorb, nele, noA, noB = f["sorb"], f["nele"], f["noA"], f["noB"]
    lut = table(f["ci"], sorb, seed=3)
    h1e, h2e = dev(f["h1e"]), dev(f["h2e"])
    H = sample_space_hamiltonian(lut.bra_key, h1e, h2e, lut, sorb, nele, noA, noB)
    e, C, info = sample_space_ground_state(lut, h1e, h2e, sorb, nele, noA, noB, nroots=3, H=H)
    assert info["converged"]
    np.testing.assert_allclose(e.cpu().numpy(), FE2S2_CI_LOWEST, rtol=0, atol=1e-9)
    s2 = spin_square(lut, C, sorb).cpu().numpy()
    s = nearest_s(s2)
    assert np.abs(s2 - s * (s + 1)).max() <= 1e-8
    # the host values: eigsh on the host matrix, <S^2> with the host closed form
    Hh = scipy.sparse.csr_matrix((H.values().cpu().numpy(), H.col_indices().cpu().numpy(), H.crow_indices().cpu().numpy()),
                                 shape=(18496, 18496))
    w, U = scipy.sparse.linalg.eigsh(Hh, k=3, which="SA", tol=1e-12)
    U = U[:, np.argsort(w)]
    key = lut.bra_key.cpu().numpy()
    s2h = np.einsum("ij,ij->j", U, closed_form(key, key, sorb) @ U)
    np.testing.assert_allclose(s2, s2h, rtol=0, atol=1e-8)
    assert s.tolist() == FE2S2_CI_SPINS


# ---- spin-targeted roots ------------------------------------------------------------------------------------------
def penalty_shift(s2_values, ss, width):
    """a shift that puts every sector other than ss more than H's spectral width above it"""
    gap = min((v - ss) ** 2 for v in set(s2_values) if abs(v - ss) > 0.5)
    return 2.0 * width / gap


@gpu
@pytest.mark.parametrize("ss", [0.0, 2.0, 6.0])
def test_full_space_spin_targeted_root(ss):
    _need_gpu()
    dets = space(12, 3, 3)
    keys = to_u8(dets, 12)
    h1e, h2e = S.random_packed_integrals(12, seed=21, symmetric=True)
    lut = table(keys, 12)
    key = lut.bra_key.cpu().numpy()
    Hd = O.hij(key, key, h1e, h2e, 12, 6)
    w, U = np.linalg.eigh(Hd)
    s2 = np.einsum("ij,ij->j", U, closed_form(key, key, 12) @ U)
    s = nearest_s(s2)
    assert np.abs(s2 - s * (s + 1)).max() < 1e-9  # the dense eigenvectors have definite spin
    want = w[np.abs(s2 - ss) < 1e-6].min()
    shift = penalty_shift(np.round(s2, 6).tolist(), ss, w[-1] - w[0])
    e, C, info = sample_space_ground_state(lut, dev(h1e), dev(h2e), 12, 6, 3, 3, spin_shift=shift, ss=ss)
    assert info["converged"]
    assert abs(float(e[0]) - want) <= 1e-9
    assert abs(info["s2"][0] - ss) <= 1e-9
    # H + shift S^2 without a target: the lowest spins come first (here the shift of the ss = 2 case and above)
    if ss == 0.0:
        e0, _, info0 = sample_space_ground_state(lut, dev(h1e), dev(h2e), 12, 6, 3, 3, spin_shift=shift)
        assert info0["converged"] and abs(info0["s2"][0]) <= 1e-9 and abs(float(e0[0]) - want) <= 1e-9
    with pytest.raises(ValueError):
        sample_space_ground_state(lut, dev(h1e), dev(h2e), 12, 6, 3, 3, ss=ss)
    with pytest.raises(ValueError):
        sample_space_ground_state(lut, dev(h1e), dev(h2e), 12, 6, 3, 3, spin_shift=-1.0)


@gpu
def test_fe2s2_ci_first_spin_rung():
    """the lowest state of the first spin, in energy order, that is not the ground state's: Davidson on
    H + shift (S^2 - ss)^2 against host eigsh on the same operator"""
    _need_gpu()
    f = fe2s2()
    sorb, nele, noA, noB = f["sorb"], f["nele"], f["noA"], f["noB"]
    lut = table(f["ci"], sorb, seed=3)
    h1e, h2e = dev(f["h1e"]), dev(f["h2e"])
    H = sample_space_hamiltonian(lut.bra_key, h1e, h2e, lut, sorb, nele, noA, noB)
    root = next(i for i, s in enumerate(FE2S2_CI_SPINS) if s != FE2S2_CI_SPINS[0])
    ss = FE2S2_CI_SPINS[root] * (FE2S2_CI_SPINS[root] + 1)
    # every other sector lies at or above the ground energy and gets a penalty of at least shift * gap: ten times the
    # target root's distance from the ground state puts all of them above it.  (A larger shift selects the same state but
    # slows Davidson down: its diagonal preconditioner does not see the penalty's spin-exchange couplings.)
    gap = min((v * (v + 1) - ss) ** 2 for v in range(3) if v != FE2S2_CI_SPINS[root])
    shift = 10.0 * (FE2S2_CI_LOWEST[root] - FE2S2_CI_LOWEST[0]) / gap
    e, C, info = sample_space_ground_state(lut, h1e, h2e, sorb, nele, noA, noB, H=H, spin_shift=shift, ss=ss)
    assert info["converged"]
    assert abs(info["s2"][0] - ss) <= 1e-8
    Hh = scipy.sparse.csr_matrix((H.values().cpu().numpy(), H.col_indices().cpu().numpy(), H.crow_indices().cpu().numpy()),
                                 shape=(18496, 18496))
    key = lut.bra_key.cpu().numpy()
    P = closed_form(key, key, sorb) - ss * scipy.sparse.identity(18496, format="csr")
    w, U = scipy.sparse.linalg.eigsh(Hh + shift * (P @ P), k=1, which="SA", tol=1e-12)
    assert abs(float(e[0]) - w[0]) <= 1e-9
    assert abs(float(e[0]) - float(U[:, 0] @ (Hh @ U[:, 0]))) <= 1e-9
    # a root of H below it has another spin, so it is the lowest of its spin: the first rung of the ladder
    assert abs(float(e[0]) - FE2S2_CI_LOWEST[root]) <= 1e-9
