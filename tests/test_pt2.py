"""Epstein-Nesbet PT2 correction of sample-space states: energy.sample_space_pt2 (pynqs_pt2_*, C_extension.pt2_sums).

  E_PT2[r] = (1 / sum_i C[i, r]^2) sum over the externals a of (sum_i <key_i|H|a> C[i, r])^2 / (E[r] - <a|H|a>)

On full small sectors the reference is the dense oracle.hij matrix of the sector; on the Fe2S2 CI space, a larger table and
multi-word ONVs it is a route through the library's existing operators (get_comb_hij_fused, WavefunctionLUT.lookup,
torch.unique, index_add_, get_hij_torch)."""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from pynqs_b200 import C_extension as ops
from pynqs_b200 import _lib
from pynqs_b200 import synthetic as S
from pynqs_b200.energy import sample_space_ground_state, sample_space_pt2
from pynqs_b200.lut import WavefunctionLUT

from test_spin_square import space, to_u8
from util import fe2s2

DEV = "cuda:0"
gpu = pytest.mark.gpu


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


# ---- host reference ------------------------------------------------------------------------------------------------------
def dense_pt2(dets, in_table, c, E, H):
    """sum over the externals a (not in the table, connected to a table row) of (H[a, T] c)^2 / (c c) / (E - H_aa), from the
    dense sector matrix H (rows / columns = dets); c [|T|, k] over the table's dets in dets order, E [k]"""
    T = np.flatnonzero(in_table)
    out = np.zeros(c.shape[1])
    for a in np.flatnonzero(~in_table):
        if not any(bin(dets[a] ^ dets[t]).count("1") <= 4 for t in T):
            continue
        out += (H[a, T] @ c) ** 2 / (E - H[a, a])
    return out / (c * c).sum(0)


def test_dense_reference_on_one_missing_determinant():
    """a whole sector minus one determinant d has exactly one external: E_PT2 = (H[d, T] c)^2 / (c c) / (E0 - H_dd)"""
    sorb, na, nb = 10, 3, 2
    dets = sorted(space(sorb, na, nb))
    h1e, h2e = S.random_packed_integrals(sorb, seed=5, symmetric=True)
    u8 = to_u8(dets, sorb)
    H = O.hij(u8, u8, h1e, h2e, sorb, na + nb)
    d = 17
    in_table = np.ones(len(dets), dtype=bool)
    in_table[d] = False
    T = np.flatnonzero(in_table)
    w, v = np.linalg.eigh(H[np.ix_(T, T)])
    c, E0 = v[:, :1], w[:1]
    got = dense_pt2(dets, in_table, c, E0, H)
    num = sum(H[d, t] * c[j, 0] for j, t in enumerate(T))
    want = num * num / float(c[:, 0] @ c[:, 0]) / (E0[0] - H[d, d])
    assert abs(got[0] - want) <= 1e-14 * abs(want)
    assert want < 0


def test_pass_count_rule():
    lg = ops.pt2_log2_parts
    assert lg(1000, 1 << 30, lambda p: 80 * p) == 0
    # 10^6 rows x 7875 excitations at 80 bytes a pair in 16 GiB: 2^6 passes of 1.23e8 pairs (9.8 GB)
    assert lg(10**6 * 7875, 16 << 30, lambda p: 80 * p) == 6
    assert lg(10**6 * 7875, 20 * 10**9, lambda p: 80 * p + (4 << 20)) == 5
    # the budget is an inclusive bound
    assert lg(1 << 20, 80 << 18, lambda p: 80 * p) == 2
    assert lg(1 << 20, (80 << 18) - 1, lambda p: 80 * p) == 3
    # a pass stays below 2^31 pairs whatever the budget
    assert lg((1 << 31) - 1, 1 << 62, lambda p: 0) == 0
    assert lg(1 << 31, 1 << 62, lambda p: 0) == 1
    assert lg(1 << 34, 1 << 62, lambda p: 0) == 4
    with pytest.raises(ValueError):
        lg(1000, 100, lambda p: 80 * p + 1000)


def test_pt2_bad_arguments_on_the_cpu():
    lib = _lib.load()
    p = _lib.vp(256)  # never dereferenced: the checks come first
    null = _lib.vp(None)
    i64 = _lib.i64

    def count(key=p, N=10, sorb=40, na=15, nb=15, gw=p, part=0, lg=0, sc=p, off=p):
        return lib.pynqs_pt2_count(key, i64(N), int(sorb), int(na), int(nb), gw, int(part), int(lg), sc, i64(1 << 30), off, null)

    def emit(key=p, N=10, h1e=p, prep=p, sorb=40, na=15, nb=15, gw=p, part=0, lg=0, off=p, pairs=100, sc=p):
        return lib.pynqs_pt2_emit(key, i64(N), h1e, prep, int(sorb), int(na), int(nb), gw, int(part), int(lg), off, i64(pairs), sc,
                                  i64(1 << 30), null)

    def reduce(N=10, pairs=100, h1e=p, h2e=p, sorb=40, nele=30, C=p, ldc=3, k=3, E=p, sc=p, acc=p):
        return lib.pynqs_pt2_reduce(i64(N), i64(pairs), h1e, h2e, int(sorb), int(nele), C, i64(ldc), int(k), E, sc, i64(1 << 30), acc, null,
                                    null)

    for bad in (dict(N=0), dict(N=1 << 31), dict(sorb=41), dict(sorb=194), dict(na=21), dict(nb=-1), dict(part=1), dict(part=-1),
                dict(lg=32), dict(lg=3, part=8), dict(key=null), dict(gw=null), dict(sc=null), dict(off=null)):
        assert count(**bad) == _lib.EVALUE, bad
    for bad in (dict(h1e=null), dict(prep=null), dict(pairs=-1), dict(pairs=1 << 31), dict(sc=null), dict(part=2, lg=1)):
        assert emit(**bad) == _lib.EVALUE, bad
    for bad in (dict(k=0), dict(k=9), dict(ldc=2), dict(nele=41), dict(N=-1), dict(pairs=-1), dict(h1e=null), dict(h2e=null),
                dict(C=null), dict(E=null), dict(sc=null), dict(acc=null), dict(sorb=0)):
        assert reduce(**bad) == _lib.EVALUE, bad
    assert b"pt2_reduce" in lib.pynqs_last_error()
    assert lib.pynqs_pt2_sort(i64(10), i64(-1), 40, p, i64(1 << 30), null) == _lib.EVALUE
    assert lib.pynqs_pt2_sort(i64(10), i64(5), 40, null, i64(1 << 30), null) == _lib.EVALUE
    nb = _lib.ctypes.c_int64()
    assert lib.pynqs_pt2_scratch_bytes(i64(10), i64(-1), 40, _lib.ctypes.byref(nb)) == _lib.EVALUE
    assert lib.pynqs_pt2_scratch_bytes(i64(0), i64(5), 40, _lib.ctypes.byref(nb)) == _lib.EVALUE
    assert lib.pynqs_pt2_scratch_bytes(i64(10), i64(5), 40, null) == _lib.EVALUE


# ---- device ----------------------------------------------------------------------------------------------------------------
def table(keys, sorb, seed=1):
    return WavefunctionLUT(dev(keys), dev(S.random_psi(keys.shape[0], seed=seed)), sorb, DEV, rank=0, world_size=1)


def ints_of(u8):
    w = u8.view(np.uint64).reshape(u8.shape[0], -1)
    return [sum(int(v) << (64 * k) for k, v in enumerate(row)) for row in w]


def ops_route(lut, C, E, h1e, h2e, sorb, nele, na, nb, chunk=1024):
    """E_PT2 from the library's existing operators: the excitations of every row (get_comb_hij_fused, chunked), the table
    members dropped (WavefunctionLUT.lookup), the externals made unique (torch.unique, return_inverse), the numerators by
    index_add_ and the diagonal by get_hij_torch.  Returns (e_pt2 [k], externals, pairs)."""
    keys = lut.bra_key
    N, W = keys.shape
    xs, hs, rows = [], [], []
    for b in range(0, N, chunk):
        comb, hmat = ops.get_comb_hij_fused(keys[b : b + chunk].contiguous(), h1e, h2e, sorb, nele, na, nb)
        m = comb.size(1) - 1
        x = comb[:, 1:].reshape(-1, W).contiguous()
        _, miss, _ = lut.lookup(x)
        xs.append(x[miss])
        hs.append(hmat[:, 1:].reshape(-1)[miss])
        rows.append(b + miss // m)
    x, h, row = torch.cat(xs), torch.cat(hs), torch.cat(rows)
    words = x.view(torch.int64)
    if W == 8:
        uniq, inv = torch.unique(words.view(-1), return_inverse=True)
    else:
        uniq, inv = torch.unique(words.view(-1, W // 8), dim=0, return_inverse=True)
    ext = uniq.contiguous().view(torch.uint8).view(-1, W)
    U = ext.size(0)
    num = torch.zeros(U, C.size(1), dtype=torch.float64, device=DEV).index_add_(0, inv, h.unsqueeze(1) * C[row])
    haa = ops.get_hij_torch(ext, ext.view(U, 1, W), h1e, h2e, sorb, nele).view(U)
    e = (num * num / (E.view(1, -1) - haa.view(-1, 1))).sum(0) / (C * C).sum(0)
    return e, U, x.size(0)


def assert_rel(got, want, rtol):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert np.all(np.abs(got - want) <= rtol * np.abs(want)), (got, want)


@gpu
@pytest.mark.parametrize("nroots", [1, 3])
@pytest.mark.parametrize("frac", [2, 4])
@pytest.mark.parametrize("sorb,na,nb", [(10, 3, 2), (12, 3, 3), (14, 4, 2)])
def test_matches_dense_reference(sorb, na, nb, frac, nroots):
    _need_gpu()
    dets = sorted(space(sorb, na, nb))
    h1e_np, h2e_np = S.random_packed_integrals(sorb, seed=sorb + frac, symmetric=True)
    u8 = to_u8(dets, sorb)
    H = O.hij(u8, u8, h1e_np, h2e_np, sorb, na + nb)
    rng = np.random.default_rng(sorb * 10 + frac)
    pick = sorted(rng.permutation(len(dets))[: len(dets) // frac])
    lut = table(u8[pick], sorb)
    h1e, h2e = dev(h1e_np), dev(h2e_np)
    e, C, info = sample_space_ground_state(lut, h1e, h2e, sorb, na + nb, na, nb, nroots, tol=1e-10)
    assert info["converged"]
    got, ginfo = sample_space_pt2(lut, C, e, h1e, h2e, sorb, na + nb, na, nb)
    assert got.dtype == torch.float64 and got.shape == (nroots,)
    # the table's dets in table order, as rows of the dense matrix
    index = {d: i for i, d in enumerate(dets)}
    order = [index[d] for d in ints_of(lut.bra_key.cpu().numpy())]
    in_table = np.zeros(len(dets), dtype=bool)
    in_table[order] = True
    Cd = np.zeros((len(dets), nroots))
    Cd[order] = C.cpu().numpy()
    want = dense_pt2(dets, in_table, Cd[in_table], e.cpu().numpy(), H)
    assert_rel(got.cpu().numpy(), want, 1e-12)
    ext = [a for a in np.flatnonzero(~in_table) if any(bin(dets[a] ^ dets[t]).count("1") <= 4 for t in order)]
    assert ginfo["externals"] == len(ext)
    assert ginfo["pairs"] == sum(bin(dets[a] ^ dets[t]).count("1") <= 4 for a in ext for t in order)
    assert ginfo["passes"] == 1


@gpu
@pytest.mark.parametrize("sorb,na,nb", [(10, 3, 2), (12, 3, 3), (14, 4, 2)])
def test_whole_sector_has_no_externals(sorb, na, nb):
    _need_gpu()
    lut = table(to_u8(space(sorb, na, nb), sorb), sorb)
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(sorb, seed=3, symmetric=True))
    e, C, _ = sample_space_ground_state(lut, h1e, h2e, sorb, na + nb, na, nb, 2)
    got, info = sample_space_pt2(lut, C, e, h1e, h2e, sorb, na + nb, na, nb)
    assert got.tolist() == [0.0, 0.0]
    assert info["externals"] == 0 and info["pairs"] == 0


@gpu
def test_fe2s2_ci_space_three_roots():
    _need_gpu()
    f = fe2s2()
    sorb, nele, na, nb = f["sorb"], f["nele"], f["noA"], f["noB"]
    lut = table(f["ci"], sorb, seed=3)
    assert lut.bra_key.size(0) == 18496
    h1e, h2e = dev(f["h1e"]), dev(f["h2e"])
    e, C, info = sample_space_ground_state(lut, h1e, h2e, sorb, nele, na, nb, 3)
    assert info["converged"]
    got, ginfo = sample_space_pt2(lut, C, e, h1e, h2e, sorb, nele, na, nb)
    want, U, pairs = ops_route(lut, C, e, h1e, h2e, sorb, nele, na, nb)
    assert_rel(got.cpu().numpy(), want.cpu().numpy(), 1e-10)
    assert ginfo["externals"] == U and ginfo["pairs"] == pairs
    # (E_PT2 of this space is positive: it leaves 6 of the 40 spin orbitals empty, and 667 432 of its externals lie below
    #  E_var, two of them within 1e-6 Ha -- intruders; DESIGN.md 4.13)


@gpu
def test_uniform_fe2s2_table_of_2e4_samples():
    _need_gpu()
    import bench

    h1e_np, h2e_np, _ = bench.load_integrals()
    sorb, nele, na, nb = bench.SORB, bench.NELE, bench.NOA, bench.NOB
    lut = table(bench.make_table("uniform", 20_000), sorb, seed=5)
    h1e, h2e = dev(h1e_np), dev(h2e_np)
    e, C, info = sample_space_ground_state(lut, h1e, h2e, sorb, nele, na, nb)
    assert info["converged"]
    got, ginfo = sample_space_pt2(lut, C, e, h1e, h2e, sorb, nele, na, nb)
    want, U, pairs = ops_route(lut, C, e, h1e, h2e, sorb, nele, na, nb)
    assert_rel(got.cpu().numpy(), want.cpu().numpy(), 1e-10)
    assert ginfo["externals"] == U and ginfo["pairs"] == pairs


@gpu
@pytest.mark.parametrize("sorb", [100, 140])
def test_multi_word_onvs(sorb):
    """Two- and three-word ONVs: 7 orbitals placed across the words, a table of two determinants and their singles and
    doubles within the 7 orbitals; the externals reach every orbital of the wide space"""
    _need_gpu()
    small, na, nb = 14, 3, 2
    pos = [1, 20, 31, 32, 40, 55, 69][: small // 2] if sorb == 140 else [0, 15, 31, 32, 33, 47, 49]
    dets = sorted(space(small, na, nb))
    base = [dets[5], dets[-9]]
    near = sorted({d for d in dets for b in base if bin(d ^ b).count("1") <= 4})

    def widen(d):
        return sum(1 << (2 * pos[k] + s) for k in range(small // 2) for s in range(2) if (d >> (2 * k + s)) & 1)

    lut = table(to_u8(sorted(widen(d) for d in near), sorb), sorb)
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(sorb, seed=9, symmetric=True))
    e, C, info = sample_space_ground_state(lut, h1e, h2e, sorb, na + nb, na, nb, 2)
    assert info["converged"]
    got, ginfo = sample_space_pt2(lut, C, e, h1e, h2e, sorb, na + nb, na, nb)
    want, U, pairs = ops_route(lut, C, e, h1e, h2e, sorb, na + nb, na, nb)
    assert_rel(got.cpu().numpy(), want.cpu().numpy(), 1e-10)
    assert ginfo["externals"] == U and ginfo["pairs"] == pairs


@gpu
def test_passes_determinism_and_column_slices():
    _need_gpu()
    import bench

    h1e_np, h2e_np, _ = bench.load_integrals()
    sorb, nele, na, nb = bench.SORB, bench.NELE, bench.NOA, bench.NOB
    lut = table(bench.make_table("zipf0.8", 3000), sorb, seed=6)
    h1e, h2e = dev(h1e_np), dev(h2e_np)
    e, C, _ = sample_space_ground_state(lut, h1e, h2e, sorb, nele, na, nb, 2)
    one, i1 = sample_space_pt2(lut, C, e, h1e, h2e, sorb, nele, na, nb)
    assert i1["passes"] == 1
    N = lut.bra_key.size(0)
    nb_ = _lib.ctypes.c_int64()
    upper = N * ops.get_Num_SinglesDoubles(sorb, na, nb)
    _lib.check(_lib.load().pynqs_pt2_scratch_bytes(_lib.i64(N), _lib.i64(-(-upper // 8)), sorb, _lib.ctypes.byref(nb_)))
    many, i8 = sample_space_pt2(lut, C, e, h1e, h2e, sorb, nele, na, nb, max_bytes=nb_.value)
    assert i8["passes"] >= 8
    assert i8["externals"] == i1["externals"] and i8["pairs"] == i1["pairs"]
    assert_rel(many.cpu().numpy(), one.cpu().numpy(), 1e-12)
    again, _ = sample_space_pt2(lut, C, e, h1e, h2e, sorb, nele, na, nb, max_bytes=nb_.value)
    assert again.cpu().numpy().tobytes() == many.cpu().numpy().tobytes()
    # k = 10: two column slices of the kernel, each column as in its own call
    rng = np.random.default_rng(8)
    C10 = dev(rng.standard_normal((N, 10)))
    E10 = e[0] - dev(rng.uniform(0.5, 2.0, 10))
    acc, _ = ops.pt2_sums(lut.bra_key, C10, E10, h1e, h2e, sorb, nele, na, nb)
    for r in range(10):
        acc_r, _ = ops.pt2_sums(lut.bra_key, C10[:, r : r + 1], E10[r : r + 1], h1e, h2e, sorb, nele, na, nb)
        assert acc_r.cpu().numpy().tobytes() == acc[r : r + 1].cpu().numpy().tobytes()
    full, _ = sample_space_pt2(lut, C10, E10, h1e, h2e, sorb, nele, na, nb)
    assert_rel(full.cpu().numpy(), (acc / (C10 * C10).sum(0)).cpu().numpy(), 1e-15)


@gpu
def test_value_errors_and_one_row_table():
    _need_gpu()
    sorb, na, nb = 12, 3, 3
    dets = space(sorb, na, nb)
    lut = table(to_u8(dets, sorb)[:100], sorb)
    h1e, h2e = (dev(a) for a in S.random_packed_integrals(sorb, seed=4, symmetric=True))
    c = lut.wf_value
    E = torch.tensor([-1.0], dtype=torch.float64, device=DEV)
    args = (h1e, h2e, sorb, na + nb, na, nb)
    with pytest.raises(ValueError):
        sample_space_pt2(lut, c.float(), E, *args)  # dtype
    with pytest.raises(ValueError):
        sample_space_pt2(lut, c[:99], E, *args)  # rows
    with pytest.raises(ValueError):
        sample_space_pt2(lut, c.view(10, 10), E, *args)  # shape
    with pytest.raises(ValueError):
        sample_space_pt2(lut, torch.stack([c, c], 1), E, *args)  # energies of the wrong length
    with pytest.raises(ValueError):
        sample_space_pt2(lut, torch.stack([c, torch.zeros_like(c)], 1), E.repeat(2), *args)  # a zero column
    with pytest.raises(ValueError):
        sample_space_pt2(lut, c, E, h1e.float(), h2e.float(), sorb, na + nb, na, nb)  # integrals
    keys = lut.bra_key.cpu().numpy()
    dup = table(np.concatenate([keys[:50], keys[40:60]]), sorb)
    with pytest.raises(ValueError, match="duplicate"):
        sample_space_pt2(dup, dup.wf_value, E, *args)
    empty = table(keys[:0], sorb)
    with pytest.raises(ValueError, match="empty"):
        sample_space_pt2(empty, empty.wf_value, E, *args)
    # one row: every single and double of it is an external, reached once
    one = table(keys[7:8], sorb)
    cc = torch.tensor([-0.5], dtype=torch.float64, device=DEV)
    got, info = sample_space_pt2(one, cc, E, *args)
    want, U, pairs = ops_route(one, cc.view(1, 1), E, *args)
    assert info["externals"] == U == pairs == info["pairs"] == ops.get_Num_SinglesDoubles(sorb, na, nb)
    assert_rel(got.cpu().numpy(), want.cpu().numpy(), 1e-12)
