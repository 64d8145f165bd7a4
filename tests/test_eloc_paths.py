"""One-pass E_loc and the sample-space Hamiltonian on the paths the small-table tests do not reach:
  A. every evaluation kernel (warp per sample, 32 samples per warp with its hand-off of long hit lists) for one-, two- and
     three-word ONVs, real and complex psi, clean tables and tables with duplicate keys;
  B. two- and three-word calls large enough for the default tuning to pick the 32-samples-per-warp kernel;
  C. calls of more samples than one batch of the per-sample route (the launchers' loop over batches);
  D. calls whose hit lists need more than the hit buffer holds (samples fall back to the reference's route mid-call).
References: the CPU oracle (the reference arithmetic) on every sample or a subsample, the three-call path
(get_comb_hij_fused -> wavefunction_lut -> reduce) on every sample, dense get_hij_torch rows bit for bit."""
import ctypes
import itertools

import numpy as np
import pytest
import scipy.sparse
import torch

from oracle import oracle as O
from pynqs_b200 import C_extension as ops
from pynqs_b200 import _lib
from pynqs_b200 import synthetic as S
from pynqs_b200.energy import local_energy_three_call
from pynqs_b200.lut import WavefunctionLUT

from util import fe2s2

DEV = "cuda:0"
gpu = pytest.mark.gpu
# E_loc of the larger tables sums tens to hundreds of O(1) terms of both signs (random psi ratios).  A few samples in 10^4
# land within 1e-13 of zero, where the kernels' and the references' summation orders differ by a few ulps of the terms
# (up to 4.4e-15 seen): those comparisons get this absolute tolerance on top of rtol = 1e-12
CANCEL_ATOL = 1e-14
HEAVY = 256  # kHeavyHits (eloc_scan.cu): a sample with more hits leaves the 32-samples-per-warp kernel for a warp of its own
TILE_MIN = 148 * 32 * 8  # calls of at least this many samples (per batch) take the 32-samples-per-warp kernel by default


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.fixture(autouse=True)
def _default_tuning():
    _lib.set_tuning()
    yield
    _lib.set_tuning()


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")


def tune(**knobs):
    _lib.set_tuning()
    for k, v in knobs.items():
        _lib.set_tuning(k, v)


_integrals = {}


def integrals(sorb):
    """seeded packed integrals, on the host and the device (1.3 GB at 192 spin orbitals: made once per module)"""
    if sorb not in _integrals:
        h1e, h2e = S.random_packed_integrals(sorb, seed=sorb + 1, symmetric=True)
        _integrals[sorb] = (h1e, h2e, dev(h1e), dev(h2e))
    return _integrals[sorb]


# ---- host-side bookkeeping ------------------------------------------------------------------------------------------
def levels(x, keys):
    """excitation level between every row of x and every key (uint8 [*, 8L]): popcount of the XOR over 2"""
    xw = np.ascontiguousarray(x).view(np.uint64)
    kw = np.ascontiguousarray(keys).view(np.uint64)
    out = np.empty((xw.shape[0], kw.shape[0]), dtype=np.int32)
    for i in range(0, xw.shape[0], 64):
        d = np.zeros((min(64, xw.shape[0] - i), kw.shape[0]), dtype=np.int32)
        for w in range(kw.shape[1]):
            d += np.bitwise_count(xw[i : i + 64, None, w] ^ kw[None, :, w])
        out[i : i + 64] = d // 2
    return out


def hits_of(x, keys):
    """(connected keys of every sample in the table, of which single excitations, copies of the sample itself): what the
    scan hands to the evaluation kernels on the full-key route"""
    lvl = levels(x, keys)
    return ((lvl == 1) | (lvl == 2)).sum(1), (lvl == 1).sum(1), (lvl == 0).sum(1)


def excitations(x, sorb, noA, noB):
    """singles and doubles of one determinant (uint8 [8L]), each [*, 8L]"""
    exc = O.comb(x[None], sorb, noA, noB)[0, 1:]
    lvl = levels(x[None], exc)[0]
    return exc[lvl == 1], exc[lvl == 2]


def drop_rows(a, b):
    """the rows of a that are not rows of b"""
    bad = {r.tobytes() for r in b}
    return a[np.array([r.tobytes() not in bad for r in a], dtype=bool)]


def cluster_table(sorb, noA, noB, n, n_seeds, seed):
    """n unique keys in random order: n_seeds random determinants and random excitations of them, about n / n_seeds per seed,
    so each seed has hundreds of connected keys in the table.  Returns (keys, rows of the seeds)."""
    rng = np.random.default_rng(seed)
    seeds = S.random_onvs(n_seeds, sorb, noA, noB, seed=seed)
    per = -(-(n - n_seeds) * 21 // 20 // n_seeds)  # 5 % spare for excitations that two seeds share
    exc = O.comb(seeds, sorb, noA, noB)[:, 1:]
    pick = np.stack([rng.choice(exc.shape[1], per, replace=False) for _ in range(n_seeds)])
    picks = drop_rows(np.unique(exc[np.arange(n_seeds)[:, None], pick].reshape(-1, seeds.shape[1]), axis=0), seeds)
    del exc
    assert picks.shape[0] >= n - n_seeds
    keys = np.concatenate([seeds, picks[rng.permutation(picks.shape[0])[: n - n_seeds]]])
    perm = rng.permutation(n)
    return np.ascontiguousarray(keys[perm]), np.argsort(perm)[:n_seeds]


def scratch_bytes(n, sorb, noA, noB):
    nb = ctypes.c_int64()
    _lib.check(_lib.load().pynqs_eloc_scratch_bytes(_lib.i64(n), sorb, noA, noB, 0, ctypes.byref(nb)))
    return nb.value


def csr(x, h1e, h2e, lut, sorb, nele, noA, noB):
    crow, col, val = ops.sample_space_hamiltonian(x, h1e, h2e, sorb, nele, noA, noB, lut.bra_key, lut.group_index)
    return crow.cpu().numpy(), col.cpu().numpy(), val.cpu().numpy()


def check_rows_against_dense(crow, col, val, rows, H, landing=None, lvl=None):
    """CSR rows `rows` against dense get_hij_torch rows H: values bit for bit at the stored columns and, on a table without
    duplicate keys, zero everywhere else; with duplicates the columns are the rows the classic search lands on"""
    for k, i in enumerate(rows):
        c, v = col[crow[i] : crow[i + 1]], val[crow[i] : crow[i + 1]]
        assert (np.diff(c) > 0).all()
        np.testing.assert_array_equal(v.view(np.uint64), H[k, c].view(np.uint64))
        if landing is None:
            rest = H[k].copy()
            rest[c] = 0.0
            assert not rest.any()
        else:
            np.testing.assert_array_equal(c, np.unique(landing[lvl[k] <= 2]))


def check_identity(crow, col, val, psi_sorted, eloc, psi0, in_table, rtol=1e-12):
    """(H psi)[i] = eloc[i] psi0[i] on the rows whose sample is in the table; the others have E_loc NaN and psi0 0"""
    N = psi_sorted.shape[0]
    Hpsi = scipy.sparse.csr_matrix((val, col, crow), shape=(crow.size - 1, N)) @ psi_sorted
    want = eloc[in_table] * psi0[in_table]
    scale = rtol * np.abs(want).max()  # rows whose sum cancels: the error is that of the largest terms
    np.testing.assert_allclose(Hpsi[in_table], want, rtol=rtol, atol=scale)
    assert np.isnan(eloc[~in_table]).all() and (psi0[~in_table] == 0).all()


# ---- A. every evaluation kernel, small -------------------------------------------------------------------------------
# (sorb, noA, noB, knob): two words (the second one full at 128), three words, one full word on the full-key route
GEOMETRIES = [(100, 3, 3, None), (128, 3, 3, None), (132, 3, 2, None), (192, 4, 4, None), (64, 8, 8, "full_keys")]
_small = {}


def small_case(sorb, noA, noB):
    """3 seeds with 400 of their excitations each in the table (> 256 hits: the list of long hit lists), 8 'middle' samples
    with 6 single and 40 double excitations each in the table (a few dozen hits, singles among them: the 32-samples-per-warp
    kernel's hit loop), 22 other table keys, 2 samples that are not in the table; 35 samples in all (one warp and a partial one)"""
    key = (sorb, noA, noB)
    if key in _small:
        return _small[key]
    rng = np.random.default_rng(sorb)
    keys, seed_rows = cluster_table(sorb, noA, noB, 3 + 3 * 400, 3, seed=sorb + 7)
    seeds = keys[seed_rows]
    others = np.delete(np.arange(keys.shape[0]), seed_rows)
    mids = keys[rng.choice(others, 8, replace=False)]
    extra = []
    for m in mids:
        singles, doubles = excitations(m, sorb, noA, noB)
        extra += [singles[rng.choice(singles.shape[0], 6, replace=False)], doubles[rng.choice(doubles.shape[0], 40, replace=False)]]
    keys = np.unique(np.concatenate([keys] + extra), axis=0)
    keys = keys[rng.permutation(keys.shape[0])]
    light = drop_rows(keys[rng.choice(keys.shape[0], 40, replace=False)], np.concatenate([seeds, mids]))[:22]
    missing = drop_rows(S.random_onvs(4, sorb, noA, noB, seed=sorb + 9), keys)[:2]
    x = np.concatenate([seeds, mids, light, missing])
    cls = np.array([0] * 3 + [1] * 8 + [2] * 22 + [3] * 2)  # heavy, middle, light, missing
    perm = rng.permutation(x.shape[0])
    _small[key] = (keys, np.ascontiguousarray(x[perm]), cls[perm])
    return _small[key]


@gpu
@pytest.mark.parametrize("dup", [False, True], ids=["clean", "dup_keys"])
@pytest.mark.parametrize("cplx", [False, True], ids=["real", "complex"])
@pytest.mark.parametrize("sorb,noA,noB,knob", GEOMETRIES, ids=[f"{g[0]}sorb_{g[1]}a{g[2]}b" for g in GEOMETRIES])
def test_every_evaluator_against_the_oracle(sorb, noA, noB, knob, cplx, dup):
    """Both evaluation kernels (eval_tiles 0: one warp per sample; 2: 32 samples per warp, long hit lists and flagged samples
    handed to the warp-per-sample kernel) against the oracle on every sample, against each other, and against the Hamiltonian
    through (H psi)[i] = eloc[i] psi0[i].  Duplicate keys flag every sample for the reference's route."""
    _need_gpu()
    keys, x, cls = small_case(sorb, noA, noB)
    if dup:
        keys = np.concatenate([keys, keys[::7], keys[::31]])  # some keys two or three times, with different psi on the copies
    nele = noA + noB
    n = x.shape[0]
    # the classes the test is about, from the host
    hits, singles, selves = hits_of(x, keys)
    assert n > 32 and n % 32 != 0
    assert (hits[cls == 0] > HEAVY).all()
    assert ((hits[cls == 1] >= 24) & (hits[cls == 1] <= HEAVY) & (singles[cls == 1] >= 1)).all()
    assert (selves[cls == 3] == 0).all() and (selves[cls != 3] >= 1).all()
    psi = S.random_psi(keys.shape[0], seed=sorb + 11, complex_=cplx)
    h1e_np, h2e_np, h1e, h2e = integrals(sorb)
    order = O.sort_onv(keys)
    skeys, spsi = keys[order], psi[order]
    want = O.eloc_sample_space(x, h1e_np, h2e_np, skeys, spsi, sorb, nele, noA, noB)
    idx, found = O.lut(skeys, x)
    want_psi0 = np.where(found, spsi[np.where(found, idx, 0)], 0)
    assert (found == (cls != 3)).all() and (np.isnan(want) == ~found).all()
    lut = WavefunctionLUT(dev(keys), dev(psi), sorb, DEV, rank=0, world_size=1)
    xd = dev(x)
    got = {}
    for tiles in (0, 2):
        tune(eval_tiles=tiles, **({knob: 1} if knob else {}))
        e, p0 = ops.eloc_sample_space(xd, h1e, h2e, sorb, nele, noA, noB, lut.bra_key, lut.wf_value, lut.group_index)
        e, p0 = e.cpu().numpy(), p0.cpu().numpy()
        np.testing.assert_allclose(e, want, rtol=1e-12, atol=0, err_msg=f"eval_tiles = {tiles}")
        np.testing.assert_array_equal(p0.view(np.float64), want_psi0.view(np.float64))
        assert (np.isnan(e) == ~found).all()
        got[tiles] = e
    np.testing.assert_allclose(got[2], got[0], rtol=1e-12, atol=0)
    # the Hamiltonian on the same inputs
    crow, col, val = csr(xd, h1e, h2e, lut, sorb, nele, noA, noB)
    assert crow[-1] == col.size
    H = ops.get_hij_torch(xd, lut.bra_key, h1e, h2e, sorb, nele).cpu().numpy()
    lvl = levels(x, skeys)
    landing = O.lut(skeys, skeys)[0] if dup else None
    check_rows_against_dense(crow, col, val, range(n), H, landing, lvl)
    check_identity(crow, col, val, spsi, got[0], want_psi0, found)


# ---- B. multi-word calls at the size where the default tuning takes the 32-samples-per-warp kernel -------------------------
_large = {}


def large_case(sorb, noA, noB, n, n_seeds):
    key = (sorb, noA, noB, n)
    if key not in _large:
        keys, seed_rows = cluster_table(sorb, noA, noB, n, n_seeds, seed=sorb + 21)
        seed_hits = hits_of(keys[seed_rows], keys)[0]
        # a random 2000 of the other samples: those the 32-samples-per-warp kernel keeps that have a single among their hits
        some = np.random.default_rng(sorb).choice(np.delete(np.arange(n), seed_rows), 2000, replace=False)
        hits, singles, _ = hits_of(keys[some], keys)
        _large[key] = (keys, seed_rows, seed_hits, some[(hits <= HEAVY) & (singles >= 1)])
    return _large[key]


@gpu
@pytest.mark.parametrize("cplx", [False, True], ids=["real", "complex"])
@pytest.mark.parametrize("sorb,noA,noB,n,n_seeds", [(100, 3, 3, 45_007, 64), (132, 3, 2, 40_003, 57)], ids=["100sorb_3a3b", "132sorb_3a2b"])
def test_multiword_default_tuning_tile_kernel(sorb, noA, noB, n, n_seeds, cplx):
    """Two- and three-word ONVs, 4e4 samples that are their own table, default tuning: the 32-samples-per-warp kernel with
    partial last warp, samples of ~700 hits handed to the warp-per-sample kernel.  Every sample against the three-call path,
    24 against the oracle (the heaviest, the last partial warp, a spread)."""
    _need_gpu()
    keys, seed_rows, seed_hits, near = large_case(sorb, noA, noB, n, n_seeds)
    assert n >= TILE_MIN and n % 32 != 0
    assert (seed_hits > HEAVY).all()
    assert near.size >= 100  # samples the tile kernel keeps that have a single excitation among their hits
    nele = noA + noB
    psi = S.random_psi(n, seed=sorb + 22, complex_=cplx)
    h1e_np, h2e_np, h1e, h2e = integrals(sorb)
    lut = WavefunctionLUT(dev(keys), dev(psi), sorb, DEV, rank=0, world_size=1)
    x = dev(keys)
    e1, p1 = ops.eloc_sample_space(x, h1e, h2e, sorb, nele, noA, noB, lut.bra_key, lut.wf_value, lut.group_index)
    assert torch.equal(p1, dev(psi))
    dtype = torch.complex128 if cplx else torch.double
    e3, _, p3 = local_energy_three_call(x, h1e, h2e, lut, sorb, nele, noA, noB, dtype, batch=1024 if sorb > 128 else 2048)
    assert torch.equal(p3, p1)
    np.testing.assert_allclose(e1.cpu().numpy(), e3.cpu().numpy(), rtol=1e-12, atol=CANCEL_ATOL)
    pick = np.unique(np.concatenate([seed_rows[np.argsort(seed_hits)[-6:]], np.arange(n - min(8, n % 32), n), near[:2],
                                     np.arange(0, n, n // 12)]))
    assert pick.size >= 20
    order = O.sort_onv(keys)
    want = O.eloc_sample_space(keys[pick], h1e_np, h2e_np, keys[order], psi[order], sorb, nele, noA, noB)
    np.testing.assert_allclose(e1.cpu().numpy()[pick], want, rtol=1e-12, atol=CANCEL_ATOL)


# ---- C. more samples than one batch of the per-sample route -------------------------------------------------------------
# (name, sorb, noA, noB, knobs, batch, sample counts): the batch is the per-sample route's, clamp(2^29 / clamp(nsd / 4, 256,
# 4096), 1024, 2^18), and every count is more than one batch and less than two
BATCH_CASES = [
    ("fe2s2_zipf_full_keys", 40, 15, 15, {"full_keys": 1}, 262_144, (262_144 + 40_000 + 13, 262_144 + 5_001)),
    ("100sorb_3a3b", 100, 3, 3, {}, 131_072, (131_072 + 40_000 + 7,)),
]


@pytest.mark.parametrize("name,sorb,noA,noB,knobs,batch,ns", BATCH_CASES, ids=[c[0] for c in BATCH_CASES])
def test_batch_cases_span_two_batches(name, sorb, noA, noB, knobs, batch, ns):
    """The batch size is not exposed; the scratch size shows it.  Up to the batch, a sample adds its hit-buffer share (>= 1 KB)
    to the scratch; from the batch on, only its 8-byte diagonal element (plus 256-byte alignment).  So `batch` is exactly the
    batch, and each count of the GPU test below runs a full batch and a second, partial one."""
    tune(**knobs)
    assert scratch_bytes(batch, sorb, noA, noB) - scratch_bytes(batch - 1, sorb, noA, noB) >= 1024
    grow = scratch_bytes(2 * batch, sorb, noA, noB) - scratch_bytes(batch, sorb, noA, noB)
    assert abs(grow - 8 * batch) <= 2048
    for n in ns:
        grow = scratch_bytes(2 * n, sorb, noA, noB) - scratch_bytes(n, sorb, noA, noB)
        assert batch < n < 2 * batch and abs(grow - 8 * n) <= 2048


@gpu
@pytest.mark.parametrize("name,sorb,noA,noB,knobs,batch,ns", BATCH_CASES, ids=[c[0] for c in BATCH_CASES])
def test_calls_over_batch_boundaries(name, sorb, noA, noB, knobs, batch, ns):
    """E_loc and psi0 of every sample against the three-call path, the oracle at the batch boundary and on the heaviest samples
    of each batch; the Hamiltonian over all rows byte for byte equal to the calls on one-batch slices, dense rows at the
    boundary, (H psi) = eloc psi0 on every row.  A second, shorter count runs a last batch below the tile kernel's threshold."""
    _need_gpu()
    n = ns[0]
    if sorb == 40:
        f = fe2s2()
        import bench

        keys = bench.make_table("zipf0.8", n)
        h1e_np, h2e_np = np.ascontiguousarray(f["h1e"]), np.ascontiguousarray(f["h2e"])
        h1e, h2e = dev(h1e_np), dev(h2e_np)
    else:
        keys, _ = cluster_table(sorb, noA, noB, n, 240, seed=sorb + 31)
        h1e_np, h2e_np, h1e, h2e = integrals(sorb)
    assert keys.shape[0] == n
    nele = noA + noB
    psi = S.random_psi(n, seed=sorb + 32)
    lut = WavefunctionLUT(dev(keys), dev(psi), sorb, DEV, rank=0, world_size=1)
    x = dev(keys)  # in random order: the samples of the heavy strings are spread over both batches
    skeys, spsi = lut.bra_key.cpu().numpy(), lut.wf_value.cpu().numpy()
    tune(**knobs)
    e1, p1 = ops.eloc_sample_space(x, h1e, h2e, sorb, nele, noA, noB, lut.bra_key, lut.wf_value, lut.group_index)
    assert torch.equal(p1, dev(psi))
    e3, _, p3 = local_energy_three_call(x, h1e, h2e, lut, sorb, nele, noA, noB, batch=4096 if sorb == 40 else 2048)
    assert torch.equal(p3, p1)
    e = e1.cpu().numpy()
    np.testing.assert_allclose(e, e3.cpu().numpy(), rtol=1e-12, atol=CANCEL_ATOL)
    # the Hamiltonian: all rows in one call, and one call per batch
    crow, col, val = csr(x, h1e, h2e, lut, sorb, nele, noA, noB)
    length = np.diff(crow)
    parts = [csr(x[lo:hi], h1e, h2e, lut, sorb, nele, noA, noB) for lo, hi in ((0, batch), (batch, n))]
    np.testing.assert_array_equal(crow, np.concatenate([parts[0][0][:-1], parts[1][0] + parts[0][0][-1]]))
    assert col.tobytes() == np.concatenate([parts[0][1], parts[1][1]]).tobytes()
    assert val.tobytes() == np.concatenate([parts[0][2], parts[1][2]]).tobytes()
    del parts
    heavy = [lo + np.argsort(length[lo:hi])[-3:] for lo, hi in ((0, batch), (batch, n))]
    for h in heavy:
        assert length[h].min() > HEAVY + 1  # both batches hand samples to the warp-per-sample kernel
    rows = np.array([0, batch - 1, batch, n - 1])
    H = ops.get_hij_torch(x[dev(rows)], lut.bra_key, h1e, h2e, sorb, nele).cpu().numpy()
    check_rows_against_dense(crow, col, val, rows, H)
    check_identity(crow, col, val, spsi, e, p1.cpu().numpy(), np.ones(n, dtype=bool))
    pick = np.unique(np.concatenate([rows, *heavy]))
    want = O.eloc_sample_space(keys[pick], h1e_np, h2e_np, skeys, spsi, sorb, nele, noA, noB)
    np.testing.assert_allclose(e[pick], want, rtol=1e-12, atol=CANCEL_ATOL)
    # shorter counts: the same samples' prefix, a last batch of another size
    for m in ns[1:]:
        assert m - batch < TILE_MIN  # the last batch drops to the warp-per-sample kernel
        em, pm = ops.eloc_sample_space(x[:m], h1e, h2e, sorb, nele, noA, noB, lut.bra_key, lut.wf_value, lut.group_index)
        np.testing.assert_allclose(em.cpu().numpy(), e3[:m].cpu().numpy(), rtol=1e-12, atol=CANCEL_ATOL)
        assert torch.equal(pm, p1[:m])
        cm, colm, valm = csr(x[:m], h1e, h2e, lut, sorb, nele, noA, noB)
        np.testing.assert_array_equal(cm, crow[: m + 1])
        assert colm.tobytes() == col[: crow[m]].tobytes() and valm.tobytes() == val[: crow[m]].tobytes()


# ---- D. the hit buffer runs out -----------------------------------------------------------------------------------------
_spaces = {}


def full_space(sorb, noA, noB):
    """every determinant of the space, in random order: each sample has all nsd of its excitations in the table"""
    if (sorb, noA, noB) not in _spaces:
        k = sorb // 2
        a = [sum(1 << (2 * i) for i in c) for c in itertools.combinations(range(k), noA)]
        b = [sum(1 << (2 * i + 1) for i in c) for c in itertools.combinations(range(k), noB)]
        L = (sorb - 1) // 64 + 1
        ints = [ai | bi for ai in a for bi in b]
        words = np.array([[(v >> (64 * w)) & (2**64 - 1) for w in range(L)] for v in ints], dtype=np.uint64)
        keys = words.view(np.uint8).reshape(-1, 8 * L)
        _spaces[(sorb, noA, noB)] = np.ascontiguousarray(keys[np.random.default_rng(sorb).permutation(keys.shape[0])])
    return _spaces[(sorb, noA, noB)]


HIT_BUFFER_CASES = [
    ("24sorb_folded", 24, 6, 6, 300, {}),
    ("24sorb_full_keys", 24, 6, 6, 300, {"full_keys": 1}),
    ("24sorb_full_keys_tiles", 24, 6, 6, 300, {"full_keys": 1, "eval_tiles": 2}),
    ("66sorb_tiles0", 66, 2, 2, 200, {"eval_tiles": 0}),
    ("66sorb_tiles2", 66, 2, 2, 200, {"eval_tiles": 2}),
]


@gpu
@pytest.mark.parametrize("name,sorb,noA,noB,n,knobs", HIT_BUFFER_CASES, ids=[c[0] for c in HIT_BUFFER_CASES])
def test_exhausted_hit_buffer(name, sorb, noA, noB, n, knobs):
    """Full spaces (24 spin orbitals 6a6b, 853 776 keys; 66 spin orbitals 2a2b, 278 784 keys, two words): every sample asks for
    all nsd of its excitations, more than twice what the hit buffer of one call holds, so the samples whose hits come late take
    the reference's route.  E_loc of every sample against the three-call path, a subsample against the oracle, every row of
    the Hamiltonian full (nsd + 1 entries)."""
    _need_gpu()
    keys = full_space(sorb, noA, noB)
    nsd = O.num_sd(sorb, noA, noB)
    # eloc_scratch_layout, per-sample route: hits per sample clamp(nsd / 4, 256, 4096), buffer batch * that + 65 536 (one batch)
    per_sample = min(max(nsd // 4, 256), 4096)
    assert n <= (1 << 29) // per_sample
    cap = n * per_sample + 65536
    assert (n * nsd, cap) == {24: (545_400, 201_736), 66: (979_600, 310_336)}[sorb]
    assert n * nsd > 2 * cap
    nele = noA + noB
    psi = S.random_psi(keys.shape[0], seed=sorb + 41)
    h1e_np, h2e_np, h1e, h2e = integrals(sorb)
    lut = WavefunctionLUT(dev(keys), dev(psi), sorb, DEV, rank=0, world_size=1)
    x = dev(keys[:n])
    tune(**knobs)
    e1, p1 = ops.eloc_sample_space(x, h1e, h2e, sorb, nele, noA, noB, lut.bra_key, lut.wf_value, lut.group_index)
    assert torch.equal(p1, dev(psi[:n]))
    e3, _, p3 = local_energy_three_call(x, h1e, h2e, lut, sorb, nele, noA, noB, batch=100)
    np.testing.assert_allclose(e1.cpu().numpy(), e3.cpu().numpy(), rtol=1e-12, atol=0)
    assert torch.equal(p3, p1)
    pick = np.arange(0, n, n // 10)
    order = O.sort_onv(keys)
    want = O.eloc_sample_space(keys[pick], h1e_np, h2e_np, keys[order], psi[order], sorb, nele, noA, noB)
    np.testing.assert_allclose(e1.cpu().numpy()[pick], want, rtol=1e-12, atol=0)
    crow, col, val = csr(x, h1e, h2e, lut, sorb, nele, noA, noB)
    assert (np.diff(crow) == nsd + 1).all()
    rows = np.array([0, n // 2, n - 1])
    check_rows_against_dense(crow, col, val, rows, ops.get_hij_torch(x[dev(rows)], lut.bra_key, h1e, h2e, sorb, nele).cpu().numpy())
    check_identity(crow, col, val, lut.wf_value.cpu().numpy(), e1.cpu().numpy(), p1.cpu().numpy(), np.ones(n, dtype=bool))
