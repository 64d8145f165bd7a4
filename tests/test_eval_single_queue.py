"""Single excitations in the evaluation kernels: the passes over a hit list put them on a per-warp queue of 32 entries, which is
flushed (lane i evaluates entry i) when the next pass's singles would not fit and when the hit list ends.  Full spaces have
every single of every sample in the table, so the queue is flushed many times:
  - 12 spin orbitals, 3a3b (400 keys, 18 singles and 117 hits a sample): a tile of 32 samples holds 576 singles, and a sample's
    alpha and beta singles come in different runs, so they land in different flushes of the 32-samples-per-warp kernel;
  - 24 spin orbitals, 6a6b (853 776 keys, 72 singles and 1 818 hits a sample): more than 32 singles of ONE sample, so every
    sample takes at least three flushes of the warp-per-sample kernel (which also takes them from the tile kernel: long lists).
E_loc against the oracle at 1e-12 relative, and two calls bit for bit (the order of the additions is fixed: no atomics)."""
import itertools

import numpy as np
import pytest
import torch

from oracle import oracle as O
from pynqs_b200 import C_extension as ops
from pynqs_b200 import _lib
from pynqs_b200 import synthetic as S
from pynqs_b200.lut import WavefunctionLUT

DEV = "cuda:0"
# (sorb, noA, noB, samples evaluated): the 24-orbital call stays small enough for its hit buffer (no sample falls back to
# the reference's route, which has no queue)
SPACES = [(12, 3, 3, 400), (24, 6, 6, 40)]
_spaces = {}


@pytest.fixture(autouse=True)
def _default_tuning():
    _lib.set_tuning()
    yield
    _lib.set_tuning()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def full_space(sorb, noA, noB):
    """every determinant of the space (one-word ONVs), in a seeded random order"""
    if (sorb, noA, noB) not in _spaces:
        k = sorb // 2
        a = [sum(1 << (2 * i) for i in c) for c in itertools.combinations(range(k), noA)]
        b = [sum(1 << (2 * i + 1) for i in c) for c in itertools.combinations(range(k), noB)]
        words = np.array([ai | bi for ai in a for bi in b], dtype=np.uint64)
        keys = words.view(np.uint8).reshape(-1, 8)
        _spaces[(sorb, noA, noB)] = np.ascontiguousarray(keys[np.random.default_rng(sorb).permutation(keys.shape[0])])
    return _spaces[(sorb, noA, noB)]


@pytest.mark.gpu
@pytest.mark.parametrize("tiles", [0, 2], ids=["warp_per_sample", "tiles"])
@pytest.mark.parametrize("cplx", [False, True], ids=["real", "complex"])
@pytest.mark.parametrize("sorb,noA,noB,n", SPACES, ids=[f"{s[0]}sorb_{s[1]}a{s[2]}b" for s in SPACES])
def test_singles_over_many_flushes(sorb, noA, noB, n, cplx, tiles):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")
    keys = full_space(sorb, noA, noB)
    k = sorb // 2
    singles = noA * (k - noA) + noB * (k - noB)
    assert singles == {12: 18, 24: 72}[sorb]  # per sample, all in the table
    nele = noA + noB
    psi = S.random_psi(keys.shape[0], seed={12: 64, 24: 75}[sorb], complex_=cplx)
    h1e, h2e = S.random_packed_integrals(sorb, seed=sorb + 52, symmetric=True)
    x = keys[:n]
    order = O.sort_onv(keys)
    skeys, spsi = keys[order], psi[order]
    want = O.eloc_sample_space(x, h1e, h2e, skeys, spsi, sorb, nele, noA, noB)
    # sum of the magnitudes of each sample's terms (psi'/psi0) H: a few samples of 400 cancel to 1e-3 of it, and there the
    # kernels' and the oracle's orders of the additions differ by a few ulps of the terms
    comb, hmat = O.comb_hij_fused(x, h1e, h2e, sorb, nele, noA, noB)
    idx, found = O.lut(skeys, comb.reshape(-1, comb.shape[-1]))
    idx, found = idx.reshape(comb.shape[:2]), found.reshape(comb.shape[:2])
    assert found.all()
    mag = np.abs(hmat * spsi[idx] / spsi[idx[:, :1]]).sum(1)
    lut = WavefunctionLUT(dev(keys), dev(psi), sorb, DEV, rank=0, world_size=1)
    xd, h1d, h2d = dev(x), dev(h1e), dev(h2e)
    _lib.set_tuning("eval_tiles", tiles)
    got = []
    for _ in range(2):
        e, p0 = ops.eloc_sample_space(xd, h1d, h2d, sorb, nele, noA, noB, lut.bra_key, lut.wf_value, lut.group_index)
        got.append(e.cpu().numpy())
        np.testing.assert_array_equal(p0.cpu().numpy().view(np.float64), psi[:n].view(np.float64))
    assert (np.abs(got[0] - want) <= 1e-12 * np.abs(want) + 1e-15 * mag).all()
    assert got[0].tobytes() == got[1].tobytes()
